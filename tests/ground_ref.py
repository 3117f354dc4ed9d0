"""Independent reference for the voxel-covariance ground modes (ground_mode 1 and 2, DESIGN.md §8).

Written from the text of DESIGN §8 and the reference lines it cites (cpp:90-200), in numpy / scipy with exact rational
arithmetic where a decision depends on it; it shares no code with the oracle's ground_voxel().

  trim x/y (inclusive, non-finite dropped) -> pcl::VoxelGrid index in float32 (floor(p * inv_leaf) - min_b, ascending)
  -> voxel centroid = the float32 nearest to the exact rational mean -> ball B(q, leaf): float32 L2_Simple < r2 strictly,
  r2 = float32(leaf64^2), n > 3 -> scatter S_ab = sum d_a d_b - sum d_a sum d_b / n of d = p - q
  -> mode 1: |S_xz|, |S_yz|, |S_zz| < 0.001, key (int)(float32(qz) * 10f)
     mode 2: numpy.linalg.eigh, lmin / trace < planarity and n_z > 0.7, key floor(n.q / w) clamped to [-32768, 32767]
  -> histogram, mode bin (tie: smallest key; largest kz in mode 1 with bin_gap < 0), mode 2 selects every bin with at
  least max(1, ceil(best / 4)) voxels -> ground = union of the balls of the accepted voxels in the selected bins.

Every decision comes with its margin: the distance of the decided quantity from its threshold and the largest amount by
which the oracle's (or the kernel's) rounding could move it. A voxel whose margin is not positive sits on a boundary:
there an exact comparison with a rounded implementation is not meaningful, and the result says which voxels they are.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from fractions import Fraction

import numpy as np
from scipy.spatial import cKDTree

F32 = np.float32
U = 2.0 ** -53          # unit roundoff of double
EIG_REL = 1e-12         # lmin of the closed-form solve is within 1e-12 * trace of eigh (test_ground_reference pins it)
THR_MODE1 = 0.001       # cpp:145, a double literal
SCALE = 149             # every float32 is an integer multiple of 2^-149


def f32_round(fr: Fraction) -> np.float32:
    """The float32 nearest to the rational `fr` (ties to even)."""
    if fr == 0:
        return F32(0.0)
    neg = fr < 0
    num, den = abs(fr.numerator), fr.denominator
    e = num.bit_length() - den.bit_length()
    s = max(e - 24, -149)
    while True:
        n2, d2 = (num, den << s) if s >= 0 else (num << -s, den)
        q, r = divmod(n2, d2)
        if q >= 1 << 24 and s > -149:
            s += 1
            continue
        break
    if 2 * r > d2 or (2 * r == d2 and q & 1):
        q += 1
    v = F32(np.ldexp(float(q), s))
    return -v if neg else v


def exact_mean_f32(vals) -> np.float32:
    """float32 nearest to the exact mean of float32 values."""
    vals = np.asarray(vals, np.float32)
    s = sum(int(v) for v in (vals.astype(np.float64) * 2.0 ** SCALE))
    return f32_round(Fraction(s, len(vals) << SCALE))


def _to_int(a):
    return [int(v) for v in (np.asarray(a, np.float32).astype(np.float64) * 2.0 ** SCALE)]


def exact_scatter(p, q):
    """S (xx, xy, xz, yy, yz, zz) of the points p [n,3] float32 about q [3] float32, as exact Fractions."""
    d = [[pi - qi for pi in _to_int(p[:, k])] for k, qi in zip(range(3), _to_int(q))]
    n = p.shape[0]
    s1 = [sum(c) for c in d]
    out = []
    for a, b in ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)):
        s2 = sum(x * y for x, y in zip(d[a], d[b]))
        out.append(Fraction(s2 * n - s1[a] * s1[b], n << (2 * SCALE)))
    return out


def sym3(s6):
    xx, xy, xz, yy, yz, zz = s6
    return np.array([[xx, xy, xz], [xy, yy, yz], [xz, yz, zz]], np.float64)


def smallest_eig(s6):
    """(lmin, normal, trace, eigen-gap) by numpy.linalg.eigh, with the sign rule of DESIGN §8: n_z > 0, or n_z == 0 and
    n_y > 0, or n_z == n_y == 0 and n_x > 0."""
    w, v = np.linalg.eigh(sym3(s6))
    n = v[:, 0].copy()
    if n[2] < 0 or (n[2] == 0 and (n[1] < 0 or (n[1] == 0 and n[0] < 0))):
        n = -n
    return float(w[0]), n, float(np.sum(np.diag(sym3(s6)))), float(w[1] - w[0])


@dataclass
class GroundRef:
    raw_src: np.ndarray          # input index of every raw (trimmed) point
    voxels: np.ndarray           # [nvox, 8] float32, the layout of the ground_voxels tap
    ball_n: np.ndarray           # points in each voxel's ball
    margin: np.ndarray           # per voxel: > 0 when every decision of the voxel is exact under any rounding
    point_class: np.ndarray      # over the input: 0 trimmed, 1 cloud, 2 ground
    hist: dict = field(default_factory=dict)
    best: int | None = None      # mode bin key
    threshold: int = 0

    @property
    def boundary(self):
        return np.flatnonzero(self.margin <= 0)

    @property
    def counts(self):
        return dict(NT=len(self.raw_src), NC=int(np.sum(self.point_class == 1)), NG=int(np.sum(self.point_class == 2)),
                    NVOX=len(self.voxels))


def ground_reference(pts, *, mode, leaf, trim_x, trim_y, bin_gap=10.0, planarity=0.01, bin_width=0.5) -> GroundRef:
    pts = np.asarray(pts, np.float32)
    xyz = pts[:, :3]
    tx, ty = F32(trim_x), F32(trim_y)
    fin = np.all(np.isfinite(xyz), axis=1)
    with np.errstate(invalid="ignore"):
        keep = fin & (xyz[:, 0] >= -tx) & (xyz[:, 0] <= tx) & (xyz[:, 1] >= -ty) & (xyz[:, 1] <= ty)
    raw_src = np.flatnonzero(keep)
    raw = np.ascontiguousarray(xyz[raw_src])
    n = len(raw)
    cls = np.zeros(len(pts), np.uint8)
    if n == 0:
        return GroundRef(raw_src, np.zeros((0, 8), F32), np.zeros(0, int), np.zeros(0), cls)

    # pcl::VoxelGrid: float32 index arithmetic, leaves in ascending index order
    inv_leaf = F32(1.0) / F32(leaf)
    cell = np.floor(raw * inv_leaf).astype(np.int64)                  # float32 product, then floor
    minb = np.floor(raw.min(axis=0) * inv_leaf).astype(np.int64)
    div = np.floor(raw.max(axis=0) * inv_leaf).astype(np.int64) - minb + 1
    ijk = cell - minb
    vidx = ijk[:, 0] + ijk[:, 1] * div[0] + ijk[:, 2] * div[0] * div[1]
    order = np.argsort(vidx, kind="stable")
    uniq, start, cnt = np.unique(vidx[order], return_index=True, return_counts=True)
    nvox = len(uniq)

    # exact centroid: integer sums at scale 2^-149, rounded once to float32
    scaled = [np.array(_to_int(raw[order, k]), dtype=object) for k in range(3)]
    q = np.empty((nvox, 3), F32)
    for k in range(3):
        sums = np.add.reduceat(scaled[k], start)
        for v in range(nvox):
            q[v, k] = f32_round(Fraction(int(sums[v]), int(cnt[v]) << SCALE))

    # balls: float32 L2_Simple, strict; the kd-tree only proposes candidates with a generous radius
    r2 = F32(np.float64(F32(leaf)) ** 2)
    tree = cKDTree(raw.astype(np.float64))
    cand = tree.query_ball_point(q.astype(np.float64), float(F32(leaf)) * (1 + 1e-4) + 1e-30)
    lens = np.array([len(c) for c in cand])
    owner = np.repeat(np.arange(nvox), lens)
    flat = np.concatenate([np.asarray(c, np.int64) for c in cand]) if lens.sum() else np.zeros(0, np.int64)
    dd = raw[flat] - q[owner]                                          # float32
    sq = (dd[:, 0] * dd[:, 0] + dd[:, 1] * dd[:, 1]) + dd[:, 2] * dd[:, 2]
    inb = sq < r2
    owner, flat = owner[inb], flat[inb]
    ball_n = np.bincount(owner, minlength=nvox)
    ball_start = np.concatenate([[0], np.cumsum(ball_n)[:-1]])

    # scatter in double with a bound on the rounding of any summation order; exact where the bound reaches a threshold
    d = raw[flat].astype(np.float64) - q[owner].astype(np.float64)      # exact
    pairs = ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2))
    nz = ball_n > 0
    seg = ball_start[nz]

    def segsum(x):
        out = np.zeros(nvox)
        if len(x):
            out[nz] = np.add.reduceat(x, seg)
        return out

    m = [segsum(d[:, k]) for k in range(3)]
    ma = [segsum(np.abs(d[:, k])) for k in range(3)]
    nn = np.maximum(ball_n, 1).astype(np.float64)
    S = np.zeros((nvox, 6))
    E = np.zeros((nvox, 6))
    for j, (a, b) in enumerate(pairs):
        S[:, j] = segsum(d[:, a] * d[:, b]) - m[a] * m[b] / nn
        E[:, j] = 4 * (ball_n + 4) * U * (segsum(np.abs(d[:, a] * d[:, b])) + ma[a] * ma[b] / nn) + 1e-300

    vox = np.zeros((nvox, 8), F32)
    vox[:, :3] = q
    margin = np.full(nvox, np.inf)
    acc = np.zeros(nvox, bool)
    keys = np.zeros(nvox, np.int64)
    pl, w = float(F32(planarity)), float(F32(bin_width))
    for v in np.flatnonzero(ball_n > 3):                               # cpp:131
        s6 = S[v]
        if mode == 1:
            test = (2, 4, 5)
            over = np.array([abs(s6[j]) - THR_MODE1 for j in test])
            dist = np.abs(over) - E[v, list(test)]
            if np.any(dist <= 0):                                      # decide it exactly
                ex = exact_scatter(raw[flat[ball_start[v]:ball_start[v] + ball_n[v]]], q[v])
                over = np.array([float(abs(ex[j]) - Fraction(THR_MODE1)) for j in test])
                ok = all(abs(ex[j]) < Fraction(THR_MODE1) for j in test)
                dist = np.abs(over) - E[v, list(test)]
            else:
                ok = bool(np.all(over < 0))
            # a voxel rejected clearly by one entry does not depend on the others
            clear = (over >= 0) & (dist > 0)
            margin[v] = dist[clear].max() if clear.any() else dist.min()
            key = int(np.trunc(np.float32(q[v, 2]) * F32(10.0)))        # float32 product, truncation toward 0 (cpp:166)
            vox[v, 7] = 1.0
        else:
            lmin, nrm, tr, gap = smallest_eig(s6)
            ratio = lmin / tr if tr > 0 else np.inf
            ok = tr > 0 and ratio < pl and nrm[2] > 0.7
            vox[v, 5:8] = nrm
            off = float(nrm @ q[v].astype(np.float64))
            key = int(np.floor(off / w))
            # how far the decided quantities may move under rounding of S and of the eigen-solve
            ds = float(E[v].max()) + EIG_REL * max(tr, 0.0)
            dn = ds / gap if gap > 0 else np.inf
            mr = abs(ratio - pl) - (ds / tr if tr > 0 else np.inf)
            mz = abs(nrm[2] - 0.7) - dn
            x = off / w
            mk = abs(x - np.round(x)) - (dn * float(np.abs(q[v]).astype(np.float64).sum()) + 4 * U * abs(off)) / w
            if not tr > 0:
                margin[v] = np.inf
            elif (mr > 0 and ratio > pl) or (mz > 0 and nrm[2] < 0.7):  # rejected clearly: the key is not used
                margin[v] = max(mr if ratio > pl else -np.inf, mz if nrm[2] < 0.7 else -np.inf)
            else:
                margin[v] = min(mr, mz, mk)
        key = min(max(key, -32768), 32767)
        keys[v] = key
        vox[v, 4] = key
        acc[v] = ok
        vox[v, 3] = 1.0 if ok else 0.0

    ref = GroundRef(raw_src, vox, ball_n, margin, cls)
    ground = np.zeros(n, bool)
    if acc.any():
        ks, kc = np.unique(keys[acc], return_counts=True)
        ref.hist = dict(zip(ks.tolist(), kc.tolist()))
        top = kc.max()
        tied = ks[kc == top]
        ref.best = int(tied.max() if (mode == 1 and bin_gap < 0) else tied.min())
        ref.threshold = max(1, -(-int(top) // 4)) if mode == 2 else int(top)
        sel = set(ks[kc >= ref.threshold].tolist()) if mode == 2 else {ref.best}
        for v in np.flatnonzero(acc):
            if keys[v] in sel:
                ground[flat[ball_start[v]:ball_start[v] + ball_n[v]]] = True
    cls[raw_src] = np.where(ground, 2, 1)
    return ref
