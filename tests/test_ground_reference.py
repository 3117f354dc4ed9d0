"""The oracle's voxel-covariance ground stage (ground_mode 1 and 2, DESIGN.md §8) against the independent reference in
ground_ref.py, tap by tap, and the oracle's closed-form 3x3 eigen-solve against numpy.linalg.eigh (CPU only).

The comparisons are exact: voxel count and centroids bit for bit, accepted flags and bin keys equal, point classes and
counts equal. The reference bounds what rounding could do to every decision; each scene asserts that none of its voxels
sits within that bound, so equality is the right bar (and a test that relied on a lucky rounding would say so)."""
import ctypes as C

import numpy as np
import pytest

from dynamicslamtool_b200 import MovingObjectRemoval, Synth
from ground_ref import exact_mean_f32, ground_reference, smallest_eig
from helpers import IDENTITY_POSE, write_cfg


def run_oracle(oracle, cfg, pts, pose=IDENTITY_POSE):
    m = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    m.push_raw_cloud_and_pose(np.ascontiguousarray(pts, np.float32), pose)
    return m


def reference_for(m, pts):
    c = m.config
    return ground_reference(pts, mode=c.ground_mode, leaf=c.gp_leaf, trim_x=c.trim_x, trim_y=c.trim_y, bin_gap=c.bin_gap,
                            planarity=c.gp_planarity, bin_width=c.gp_bin_width)


def assert_matches_reference(m, ref, where, allow_boundary=False):
    """Every ground tap of the oracle handle `m` equals the reference `ref`."""
    if not allow_boundary:
        assert len(ref.boundary) == 0, f"{where}: voxels on a decision boundary: {ref.boundary[:20].tolist()}"
    vo = m.tap("ground_voxels")
    cnt = m.counts()
    decided = len(ref.boundary) == 0  # otherwise the ground set may follow the rounding of a boundary voxel
    for k, v in ref.counts.items():
        assert cnt[k] == v or (not decided and k in ("NC", "NG")), f"{where}: count {k}: oracle {cnt[k]} reference {v}"
    rv = ref.voxels
    assert np.array_equal(vo[:, :3].view(np.uint32), rv[:, :3].view(np.uint32)), \
        f"{where}: {int(np.sum(vo[:, :3] != rv[:, :3]))} centroid values differ from the exactly rounded mean"
    sure = ref.margin > 0
    bad = np.flatnonzero(sure & (vo[:, 3] != rv[:, 3]))
    assert len(bad) == 0, f"{where}: accepted flag differs in voxels {bad[:20].tolist()}"
    acc = sure & (rv[:, 3] > 0)
    bad = np.flatnonzero(acc & (vo[:, 4] != rv[:, 4]))
    assert len(bad) == 0, f"{where}: bin key differs in voxels {bad[:20].tolist()}: oracle {vo[bad[:5], 4]} reference {rv[bad[:5], 4]}"
    np.testing.assert_allclose(vo[acc, 5:], rv[acc, 5:], rtol=0, atol=1e-6, err_msg=f"{where}: normals")
    assert not decided or np.array_equal(m.tap("point_class"), ref.point_class), \
        f"{where}: point classes differ in {int(np.sum(m.tap('point_class') != ref.point_class))} points"


# ------------------------------------------------------------------ synthetic frames
@pytest.mark.parametrize("scenario,base,frame,overrides", [
    (4, "MOR_config_terrain.txt", 0, {}),                                      # C4, mode 2, leaf 0.5
    (4, "MOR_config_terrain.txt", 3, {"ground_mode": 1}),                      # C4, mode 1, leaf 0.5
    (4, "MOR_config_terrain.txt", 1, {"gp_leaf": 0.1, "trim_x": 12, "trim_y": 12}),
    (4, "MOR_config_terrain.txt", 2, {"ground_mode": 1, "gp_leaf": 0.1, "trim_x": 12, "trim_y": 12}),
    (1, "MOR_config.txt", 0, {"ground_mode": 1}),                              # C1, the reference defaults
    (1, "MOR_config.txt", 5, {"ground_mode": 2, "gp_bin_width": 0.1}),
])
def test_oracle_ground_stage_matches_reference_on_synthetic_frames(oracle, cfg_dir, tmp_path, scenario, base, frame, overrides):
    cfg = write_cfg(tmp_path, base=cfg_dir / base, **overrides)
    pts, pose = Synth(scenario, scenario).frame(frame)
    m = run_oracle(oracle, cfg, pts, pose)
    ref = reference_for(m, pts)
    assert ref.counts["NG"] > 0 and len(ref.hist) > 0
    assert_matches_reference(m, ref, f"C{scenario} frame {frame} {overrides}")


def _terrain(kind, rng):
    """Seeded scenes with several ground planes: two road levels, a kerb, a staircase; clutter on top."""
    n = 12000
    xy = rng.uniform(-9, 9, (n, 2))
    if kind == "multiplane":  # a level road and a 10 % ramp beside it
        z = np.where(xy[:, 0] < 0, -1.6, -1.6 + 0.1 * xy[:, 0])
    elif kind == "kerb":       # road and pavement 15 cm higher
        z = np.where(xy[:, 1] < 2.0, -1.6, -1.45)
    else:                      # stairs: 0.3 m treads, 0.17 m risers
        z = -1.6 + 0.17 * np.floor(np.clip(xy[:, 0], 0, None) / 0.3)
    z = z + rng.normal(0, 0.004, n)
    clutter = np.concatenate([rng.normal(c, 0.2, (400, 3)) for c in rng.uniform([-8, -8, -1], [8, 8, 0.5], (6, 3))])
    pts = np.concatenate([np.column_stack([xy, z]), clutter]).astype(np.float32)
    return np.column_stack([pts, np.full(len(pts), 0.5, np.float32)]).astype(np.float32)


@pytest.mark.parametrize("kind", ["multiplane", "kerb", "stairs"])
@pytest.mark.parametrize("mode,leaf,width", [(1, 0.5, 0.5), (2, 0.5, 0.2), (2, 0.3, 0.1)])
def test_oracle_ground_stage_matches_reference_on_random_terrain(oracle, tmp_path, kind, mode, leaf, width):
    rng = np.random.default_rng({"multiplane": 11, "kerb": 12, "stairs": 13}[kind] * 10 + mode)
    pts = _terrain(kind, rng)
    cfg = write_cfg(tmp_path, ground_mode=mode, gp_leaf=leaf, gp_bin_width=width, trim_x=10, trim_y=10)
    m = run_oracle(oracle, cfg, pts)
    ref = reference_for(m, pts)
    assert ref.counts["NG"] > 0
    if mode == 2:
        assert len(ref.hist) > 1
    assert_matches_reference(m, ref, f"{kind} mode {mode} leaf {leaf}")


def sloped_plane(z_of_x):
    """A 20 x 20 m lattice at 0.1 m spacing (float32 coordinates of multiples of 0.1)."""
    g = np.arange(-100, 100, dtype=np.float64) * 0.1
    x, y = np.meshgrid(g, g)
    return np.column_stack([x.ravel(), y.ravel(), z_of_x(x).ravel(), np.zeros(x.size)]).astype(np.float32)


def test_sloped_plane_through_origin_splits_over_two_bins(oracle, tmp_path):
    """The plane z = 0.2 x through the origin, mode 2, leaf 0.5, bin width 0.2: every voxel's plane offset n.q is 0 in exact
    arithmetic, but the float32 lattice coordinates scatter the fitted offsets over about +-1e-6, so the keys split over
    bins -1 and 0. That is a property of the mode-2 definition on float32 input, not rounding noise of the arithmetic:
    the offsets lie many orders of magnitude beyond any rounding bound (no voxel on a boundary), and every implementation
    must put each voxel in the same bin. The plane z = 0.1 x - 1.6 lands in one bin. The level plane z = -1.6 sits
    exactly on a bin boundary (float32 1.6 and 0.2 have the same significand, so q_z / w = -8 exactly): its keys are
    decided by the normal being exactly (0, 0, 1), which both the closed-form solve and eigh deliver."""
    cfg = write_cfg(tmp_path, ground_mode=2, gp_leaf=0.5, gp_bin_width=0.2, trim_x=100, trim_y=100)
    for name, fz, bins, on_boundary in (("z = 0.2x", lambda x: 0.2 * x, {-1, 0}, False),
                                        ("z = 0.1x - 1.6", lambda x: 0.1 * x - 1.6, {-8}, False),
                                        ("z = -1.6", lambda x: 0 * x - 1.6, {-8}, True)):
        pts = sloped_plane(fz)
        m = run_oracle(oracle, cfg, pts)
        ref = reference_for(m, pts)
        assert ref.counts["NVOX"] == 1600 and np.all(ref.voxels[:, 3] == 1), name
        assert set(ref.hist) == bins, f"{name}: bins {ref.hist}"
        assert len(ref.boundary) == (1600 if on_boundary else 0), name
        assert_matches_reference(m, ref, name, allow_boundary=on_boundary)
        assert np.array_equal(m.tap("ground_voxels")[:, 4], ref.voxels[:, 4]), name
        assert ref.counts["NG"] == 40000  # both bins hold more than 25 % of the mode bin


# ------------------------------------------------------------------ constructed scenes at the decision boundaries
def patch(x0, y0, z, nx, ny, leaf=0.5, per=4):
    """Level patch of nx x ny voxels of edge `leaf` from (x0, y0), `per` x `per` points per voxel, centred in their
    sub-cells (dyadic when x0, y0, z and leaf are)."""
    s = leaf / per
    g = lambda n, o: o + s / 2 + s * np.arange(n * per)  # noqa: E731
    x, y = np.meshgrid(g(nx, x0), g(ny, y0))
    return np.column_stack([x.ravel(), y.ravel(), np.full(x.size, z)])


def cloud(*parts):
    xyz = np.concatenate(parts).astype(np.float32)
    return np.ascontiguousarray(np.column_stack([xyz, np.full(len(xyz), 0.5, np.float32)]))


def _levels_mode1():
    # qz * 10 exactly 5, just below 5 (0.5 - 2^-24 and 0.5 - 2^-20: key 4), -2.5 (truncates toward 0: -2), -15
    zs = [0.5, 0.5 - 2.0 ** -24, -0.25, -1.5, 0.5 - 2.0 ** -20]
    return cloud(*[patch(-12 + 5 * i, 0, z, 2, 2) for i, z in enumerate(zs)])


def _mode2_peaks():
    # mode bin -2 with 17 voxels: threshold ceil(17/4) = 5; a 5-voxel peak (selected) and a 4-voxel peak (not)
    return cloud(patch(-10, -10, -0.9375, 17, 1), patch(0, 0, 0.3125, 5, 1), patch(6, 6, 1.3125, 4, 1))


def _ties(bin_gap):
    # two peaks of 4 voxels each, keys 2 and -3 (mode 1): the smaller key (-3) wins, the larger one with bin_gap < 0
    return cloud(patch(-8, -8, 0.25, 2, 2), patch(4, 4, -0.375, 2, 2))


def _ball_sizes():
    # voxels of two points each (centroid at the middle); a third point exactly `leaf` away is outside the strict ball
    # (3 points: not evaluated), one 2^-12 closer is inside (4 points: evaluated and accepted)
    out = []
    for i, gap in enumerate((0.0, 2.0 ** -12)):
        c = np.array([0.25 + 4 * i, 0.25, -1.0])
        out += [c + [-0.0625, 0, 0], c + [0.0625, 0, 0], c + [0.5 - gap, 0, 0], c + [0, 0.0625 - 0.5, 0]]
    # the fourth point lies 0.4375 from the centroid in y: with it the balls hold 3 and 4 points
    return cloud(np.array(out))


def _multiples_of_leaf():
    # lattice of exact multiples of the (non-dyadic) leaf 0.1, negative and positive: float32 index products
    g = np.float32(np.arange(-30, 31) * np.float32(0.1))
    x, y = np.meshgrid(g, g)
    return cloud(np.column_stack([x.ravel(), y.ravel(), np.float32(-0.3) + 0 * x.ravel()]))


SCENES = {
    "mode1_key_boundaries": (1, {}, _levels_mode1),
    "mode1_tie_smallest_key": (1, {"bin_gap": 10}, lambda: _ties(10)),
    "mode1_tie_bin_gap_negative": (1, {"bin_gap": -10}, lambda: _ties(-10)),
    "mode2_level_on_bin_boundary": (2, {"gp_bin_width": 0.25}, lambda: cloud(patch(-4, -4, -1.25, 6, 6), patch(4, 4, 0.5, 3, 3))),
    "mode2_peak_at_quarter": (2, {}, _mode2_peaks),
    "mode2_sloped_through_origin": (2, {"gp_bin_width": 0.2, "trim_x": 100, "trim_y": 100}, lambda: sloped_plane(lambda x: 0.2 * x)),
    "mode2_dyadic_slope_through_origin": (2, {"gp_bin_width": 0.125}, lambda: cloud(patch(-4, -4, 0, 16, 16) @ np.array([[1, 0, 0.25], [0, 1, 0], [0, 0, 1]]))),
    "mode2_keys_clamped": (2, {"gp_bin_width": 1e-5}, lambda: cloud(patch(-6, -6, -1.0, 3, 3), patch(4, 4, 1.0, 3, 3))),
    "mode1_ball_3_and_4_points": (1, {}, _ball_sizes),
    "mode2_ball_3_and_4_points": (2, {}, _ball_sizes),
    "mode1_multiples_of_leaf": (1, {"gp_leaf": 0.1}, _multiples_of_leaf),
    "mode2_multiples_of_leaf": (2, {"gp_leaf": 0.1, "gp_bin_width": 0.1}, _multiples_of_leaf),
    "mode1_nothing_accepted": (1, {}, lambda: cloud(np.random.default_rng(3).uniform(-2, 2, (3000, 3)))),
    "mode2_nothing_accepted": (2, {}, lambda: cloud(np.random.default_rng(3).uniform(-1, 1, (20000, 3)))),
    "mode1_all_trimmed": (1, {"trim_x": 1, "trim_y": 1}, lambda: cloud(patch(3, 3, 0, 2, 2))),
    "mode2_one_point": (2, {}, lambda: cloud(np.array([[0.25, 0.25, -1.0]]))),
}



@pytest.mark.parametrize("name", list(SCENES))
def test_oracle_ground_stage_matches_reference_on_constructed_scenes(oracle, tmp_path, name):
    """The scenes of test_gpu_ground_edges.py (keys, ties, peaks, ball sizes, float32 voxel index) on the oracle; voxels
    that sit on a boundary are compared where the reference decides them."""
    mode, kw, make = SCENES[name]
    pts = make()
    cfg = write_cfg(tmp_path, **{**dict(ground_mode=mode, gp_leaf=0.5, gp_bin_width=0.5, trim_x=50, trim_y=50), **kw})
    m = run_oracle(oracle, cfg, pts)
    ref = reference_for(m, pts)
    assert_matches_reference(m, ref, name, allow_boundary=True)


# ------------------------------------------------------------------ centroids: the exactly rounded mean
def test_exact_mean_helper():
    assert exact_mean_f32([1.0, np.float32(1 + 2 ** -23)]) == np.float32(1.0)          # tie between 1 and 1+2^-23: even
    assert exact_mean_f32([1.0, np.float32(1 + 2 ** -22)]) == np.float32(1 + 2 ** -23)
    assert exact_mean_f32([3e-40, 0.0]) == np.float32(1.5e-40)                        # subnormal
    assert exact_mean_f32([-0.1, -0.1, -0.1]) == np.float32(-0.1)


# ------------------------------------------------------------------ closed-form eigen-solve (mode 2)
def _sym3(oracle):
    f = oracle.lib.oracle_sym3_smallest_eig
    f.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]

    def solve(s6):
        a = (C.c_double * 6)(*[float(v) for v in s6])
        lmin, n = C.c_double(), (C.c_double * 3)()
        assert f(a, C.byref(lmin), n) == 0
        return lmin.value, np.array(n[:])
    return solve


def _matrices(rng):
    """(name, s6) for random SPD, exact rank-2 (plane), near-planar and diagonal matrices with repeated eigenvalues."""
    out = []
    for i in range(300):
        a = rng.normal(size=(3, 3))
        out.append(("spd", a @ a.T))
    for i in range(300):  # scatter of points on a plane through a random normal: rank 2
        nrm = rng.normal(size=3)
        nrm[2] = abs(nrm[2]) + 0.3
        u = np.cross(nrm, rng.normal(size=3))
        v = np.cross(nrm, u)
        p = rng.normal(size=(40, 1)) * u + rng.normal(size=(40, 1)) * v
        p -= p.mean(axis=0)
        out.append(("plane", p.T @ p))
    for noise in (1e-3, 1e-5, 1e-7, 1e-9):
        for i in range(100):
            p = np.column_stack([rng.uniform(-0.5, 0.5, (60, 2)), rng.normal(0, noise, 60)])
            r, _ = np.linalg.qr(rng.normal(size=(3, 3)))
            p = p @ (r if i % 2 else np.eye(3)).T
            p -= p.mean(axis=0)
            out.append((f"near-planar {noise:g}", p.T @ p))
    for d in ([1, 1, 1], [2, 2, 1], [1, 2, 2], [3, 1, 3], [0, 5, 5], [4, 4, 0], [0, 0, 0], [1e-3, 1, 1]):
        out.append((f"diag {d}", np.diag(np.asarray(d, np.float64))))
    return [(name, np.array([a[0, 0], a[0, 1], a[0, 2], a[1, 1], a[1, 2], a[2, 2]])) for name, a in out]


def test_sym3_smallest_eig_matches_eigh(oracle):
    solve = _sym3(oracle)
    checked_normals = 0
    for name, s6 in _matrices(np.random.default_rng(7)):
        lmin, n = solve(s6)
        wl, wn, tr, gap = smallest_eig(s6)
        assert abs(lmin - wl) <= 1e-12 * max(tr, 1e-300) or tr == 0, f"{name}: lmin {lmin} eigh {wl} trace {tr}"
        assert abs(np.linalg.norm(n) - 1) < 1e-12, name
        # sign rule: n_z > 0, or n_z == 0 and n_y > 0, or n_z == n_y == 0 and n_x > 0
        assert n[2] > 0 or (n[2] == 0 and (n[1] > 0 or (n[1] == 0 and n[0] > 0))), f"{name}: sign of {n}"
        if tr > 0 and gap >= 1e-6 * tr:
            ang = np.arctan2(np.linalg.norm(np.cross(n, wn)), abs(float(n @ wn)))
            assert ang <= 1e-9, f"{name}: normal {n} eigh {wn}: {ang} rad"
            assert np.array_equal(np.sign(n), np.sign(wn)) or np.any(np.abs(wn) < 1e-9), f"{name}: sign {n} vs {wn}"
            checked_normals += 1
    assert checked_normals > 1000


def test_sym3_degenerate_cases(oracle):
    solve = _sym3(oracle)
    lmin, n = solve([0, 0, 0, 0, 0, 0])            # no points spread: the rule's +z
    assert lmin == 0 and list(n) == [0, 0, 1]
    lmin, n = solve([2, 0, 0, 2, 0, 2])            # isotropic: any direction, the rule picks +z
    assert lmin == pytest.approx(2.0, abs=1e-15) and list(n) == [0, 0, 1]
    lmin, n = solve([1, 0, 0, 1, 0, 0])            # level plane: normal exactly +z
    assert abs(lmin) <= 1e-15 and n[0] == 0 and n[1] == 0 and n[2] > 0
    lmin, n = solve([0, 0, 0, 1, 0, 1])            # vertical plane x = 0: the normal has n_z = 0 and points to +x
    assert n[2] == 0 and n[1] == 0 and n[0] > 0
