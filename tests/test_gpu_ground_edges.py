"""The CUDA ground stage (ground_mode 1 and 2, csrc/mor_ground.cuh) at the decision boundaries of DESIGN §8 (-m gpu).

Constructed scenes, mostly on a dyadic lattice (coordinates that are multiples of 2^-10 and small): there every double
sum and product of the ball moments is exact in any order, so the kernel, the oracle and the reference in ground_ref.py
must agree bit for bit on centroids, accepted flags and bin keys, and on the point classes, even where a key or a flag
sits exactly on its threshold. Each scene runs on the single-handle path; two of them also through the pipelined,
batched (mor_batch_step_device) and mixed (mor_batch_step_device_mixed) steps."""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest

from dynamicslamtool_b200 import MixedBatch, MorError, MovingObjectRemoval, SequenceBatch, Synth
from ground_ref import exact_mean_f32, f32_round, ground_reference
from helpers import IDENTITY_POSE, write_cfg
from parity import compare_frame
from test_ground_reference import SCENES, cloud, patch

pytestmark = pytest.mark.gpu

ERR_CAPACITY, ERR_GROUND_CAP = 6, 8


def _cfg(tmp_path, mode, **kw):
    base = dict(ground_mode=mode, gp_leaf=0.5, gp_bin_width=0.5, trim_x=50, trim_y=50, min_cluster_size=5)
    base.update(kw)
    return write_cfg(tmp_path, f"g{mode}.txt", **base)


def run_scene(product, oracle, cfg, pts, max_cells=0):
    """GPU (single handle, unpipelined), oracle and reference on one frame."""
    gpu = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=max(len(pts), 1), max_cells=max_cells)
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    gpu.push_raw_cloud_and_pose(pts, IDENTITY_POSE)
    orc.push_raw_cloud_and_pose(pts, IDENTITY_POSE)
    c = orc.config
    ref = ground_reference(pts, mode=c.ground_mode, leaf=c.gp_leaf, trim_x=c.trim_x, trim_y=c.trim_y, bin_gap=c.bin_gap,
                           planarity=c.gp_planarity, bin_width=c.gp_bin_width)
    return gpu, orc, ref


def assert_exact(gpu, orc, ref, where):
    """GPU = oracle bit for bit on the ground taps; both = reference where the reference decides."""
    vg, vo = gpu.tap("ground_voxels"), orc.tap("ground_voxels")
    assert vg.shape == vo.shape == ref.voxels.shape, f"{where}: voxels {vg.shape} {vo.shape} {ref.voxels.shape}"
    assert np.array_equal(vg[:, :5].view(np.uint32), vo[:, :5].view(np.uint32)), \
        f"{where}: centroid / flag / key bits differ in rows {np.flatnonzero(np.any(vg[:, :5] != vo[:, :5], axis=1))[:10]}"
    np.testing.assert_allclose(vg[:, 5:], vo[:, 5:], rtol=0, atol=1e-6, err_msg=f"{where}: normals")
    assert np.array_equal(vg[:, :3].view(np.uint32), ref.voxels[:, :3].view(np.uint32)), f"{where}: centroid != exact mean"
    sure = ref.margin > 0
    assert np.array_equal(vg[sure, 3], ref.voxels[sure, 3]), f"{where}: flags differ from the reference"
    acc = sure & (ref.voxels[:, 3] > 0)
    assert np.array_equal(vg[acc, 4], ref.voxels[acc, 4]), f"{where}: keys differ from the reference"
    assert np.array_equal(gpu.tap("point_class"), orc.tap("point_class")), f"{where}: point classes differ from the oracle"
    if len(ref.boundary) == 0:
        assert np.array_equal(gpu.tap("point_class"), ref.point_class), f"{where}: point classes differ from the reference"
    cg = gpu.counts()
    assert cg["ERRFLAGS"] == 0, f"{where}: ERRFLAGS {cg['ERRFLAGS']}"
    for k, v in ref.counts.items():  # on a boundary the ground set follows the rounding the GPU shares with the oracle
        assert cg[k] == v or (len(ref.boundary) and k in ("NC", "NG")), f"{where}: count {k} gpu {cg[k]} reference {v}"
    og, oo = gpu.filter_cloud().copy(), orc.filter_cloud().copy()
    bad = compare_frame(gpu, orc, og, oo)
    assert not bad, f"{where}: {bad}"


@pytest.mark.parametrize("name", list(SCENES))
def test_ground_edge_scene(product, oracle, tmp_path, name):
    mode, kw, make = SCENES[name]
    pts = make()
    gpu, orc, ref = run_scene(product, oracle, _cfg(tmp_path, mode, **kw), pts)
    assert_exact(gpu, orc, ref, name)
    v = ref.voxels
    if name == "mode1_key_boundaries":
        assert sorted(set(v[v[:, 3] > 0, 4].tolist())) == [-15.0, -2.0, 4.0, 5.0]
    elif name.startswith("mode1_tie"):
        assert ref.best == (-3 if "smallest" in name else 2) and ref.counts["NG"] == 64
    elif name == "mode2_peak_at_quarter":
        assert ref.hist == {-2: 17, 0: 5, 2: 4} and ref.threshold == 5 and ref.counts["NG"] == 16 * 22
    elif name == "mode2_level_on_bin_boundary":
        assert len(ref.boundary) == 45  # q_z / w exactly -5 and 2: the keys follow the last bit of n_z
    elif name == "mode2_sloped_through_origin":
        assert set(ref.hist) == {-1, 0} and len(ref.boundary) == 0
    elif name == "mode2_keys_clamped":
        assert set(ref.hist) == {-32768, 32767}
    elif name.endswith("ball_3_and_4_points"):
        three, four = ref.ball_n == 3, ref.ball_n == 4
        assert three.sum() >= 1 and four.sum() == 1 and not np.any(v[three, 3]) and np.all(v[four, 3] == 1)
    elif name.endswith("nothing_accepted"):
        assert not np.any(v[:, 3]) and ref.counts["NG"] == 0
    elif name == "mode1_all_trimmed":
        assert ref.counts["NT"] == 0
    elif name == "mode2_one_point":
        assert ref.counts["NVOX"] == 1 and ref.counts["NG"] == 0


# ------------------------------------------------------------------ ERR_GROUND_CAP at max_cells and beyond
def _cells(pts, leaf):
    """Cells of the voxel table and of the ball grid for the raw box (the formulas of DESIGN §8)."""
    xyz = pts[:, :3]
    inv = np.float32(1) / np.float32(leaf)
    lo, hi = xyz.min(axis=0), xyz.max(axis=0)
    vox = np.prod(np.floor(hi * inv).astype(np.int64) - np.floor(lo * inv).astype(np.int64) + 1)
    h = float(np.float32(leaf)) * (1 + 2.0 ** -10)
    grid = np.prod(np.floor((hi.astype(np.float64) - lo.astype(np.float64)) * (1.0 / h)) + 1).astype(np.int64)
    return int(vox), int(grid)


@pytest.mark.parametrize("mode", [1, 2])
def test_ground_cap_exact_at_the_limit_flagged_beyond(product, oracle, tmp_path, mode):
    """The oracle has no cap: a frame whose voxel table needs exactly max_cells cells is exact, one cell more is
    ERR_GROUND_CAP. The ball grid (cell leaf * (1 + 2^-10)) never needs more cells than the voxel table, so the table's
    limit is the one reached; the box spans an exact multiple of the leaf, where the two differ by one per axis."""
    pts = cloud(patch(-2, -2, -1.0, 8, 8), np.array([[-2.0, -2.0, 0.0], [2.0, 2.0, -1.0]]))
    vox, grid = _cells(pts, 0.5)
    assert grid < vox
    cfg = _cfg(tmp_path, mode)
    gpu, orc, ref = run_scene(product, oracle, cfg, pts, max_cells=vox)
    assert_exact(gpu, orc, ref, f"max_cells = {vox}")
    gpu = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=len(pts), max_cells=vox - 1)
    gpu.push_raw_cloud_and_pose(pts, IDENTITY_POSE)
    assert gpu.counts()["ERRFLAGS"] & ERR_GROUND_CAP
    with pytest.raises(MorError) as e:
        gpu.filter_cloud()
    assert e.value.status == ERR_CAPACITY


# ------------------------------------------------------------------ determinism and centroids
def test_ground_voxels_run_to_run(product, cfg_dir, tmp_path):
    """Five runs of one C4 frame: flags, keys and centroids identical; normals may differ in their last bits only if the
    ball moments depend on the order of the atomics (reported)."""
    for mode in (1, 2):
        cfg = write_cfg(tmp_path, base=cfg_dir / "MOR_config_terrain.txt", ground_mode=mode)
        pts, pose = Synth(4, 4).frame(2)
        taps = []
        for _ in range(5):
            h = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=len(pts))
            h.push_raw_cloud_and_pose(pts, pose)
            taps.append(h.tap("ground_voxels").copy())
        for t in taps[1:]:
            assert np.array_equal(t[:, :5].view(np.uint32), taps[0][:, :5].view(np.uint32)), f"mode {mode}"
        print(f"mode {mode}: normal bits differing between runs:",
              [int(np.sum(t[:, 5:].view(np.uint32) != taps[0][:, 5:].view(np.uint32))) for t in taps[1:]])


def _fixed_mean_f32(vals):
    """float32 nearest to the mean of the values truncated to multiples of 2^-46 (DESIGN §6)."""
    t = np.floor(np.asarray(vals, np.float32).astype(np.float64) * 2.0 ** 46)
    return f32_round(Fraction(sum(int(v) for v in t), len(t) << 46))


def test_centroids_are_the_exactly_rounded_mean(product, oracle, tmp_path):
    """Voxel centroids (ground stage) and cluster centroids (clustering) against the exact rational mean. Coordinates that
    are multiples of 2^-46 (every float of magnitude >= 2^-23, and the dyadic ones below) give the exactly rounded mean;
    below that, the fixed-point split drops the bits under 2^-46 and the centroid is the rounded mean of the truncated
    values, which this test pins with coordinates such as 1e-9."""
    rng = np.random.default_rng(5)
    tiny = np.float32([2.0 ** -30, -(2.0 ** -40), 3 * 2.0 ** -27, 2.0 ** -24])
    blob = np.column_stack([rng.uniform(0.05, 0.45, 40), rng.uniform(0.05, 0.45, 40), rng.choice(tiny, 40)]).astype(np.float32)
    blob[:10, 0] = rng.choice(tiny, 10)
    pts = cloud(blob, blob + np.float32([1.3, 0, 0.7]))
    gpu, orc, ref = run_scene(product, oracle, _cfg(tmp_path, 1), pts)
    vg = gpu.tap("ground_voxels")
    assert np.array_equal(vg[:, :3].view(np.uint32), ref.voxels[:, :3].view(np.uint32)), "voxel centroids"

    below = blob.copy()
    below[:, 2] = rng.uniform(-3e-9, 3e-9, 40).astype(np.float32)  # not multiples of 2^-46
    pts = cloud(blob, below + np.float32([1.3, 0, 0]))
    cfg = write_cfg(tmp_path, "crop.txt", ec_distance_threshold=0.3, min_cluster_size=5, trim_x=1000, trim_y=1000, trim_z=1000, gp_limit=-1000)
    gpu = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=len(pts))
    gpu.push_raw_cloud_and_pose(pts, IDENTITY_POSE)
    cent, cid = gpu.tap("centroids"), gpu.tap("cluster_id")
    assert len(cent) == 2
    inexact = 0
    for k in range(len(cent)):
        members = pts[cid == k, :3]
        want = np.array([_fixed_mean_f32(members[:, q]) for q in range(3)], np.float32)
        assert np.array_equal(cent[k].view(np.uint32), want.view(np.uint32)), f"cluster {k}: {cent[k]} vs {want}"
        exact = np.array([exact_mean_f32(members[:, q]) for q in range(3)], np.float32)
        inexact += int(np.sum(cent[k] != exact))
    print("cluster centroid values that differ from the exactly rounded mean:", inexact)


# ------------------------------------------------------------------ the same bodies on the other step paths
WIRED = ("mode2_peak_at_quarter", "mode1_ball_3_and_4_points")


def _alloc(product, nbytes):
    p = C.c_void_p()
    assert product.device_alloc(0, max(nbytes, 16), C.byref(p)) == 0
    return p


def test_pipelined_batched_and_mixed_steps_equal_the_single_handle(product, oracle, tmp_path):
    scenes = [(SCENES[n][0], SCENES[n][1], SCENES[n][2]()) for n in WIRED]
    cfgs = [write_cfg(tmp_path, f"w{i}.txt", **{**dict(ground_mode=m, gp_leaf=0.5, gp_bin_width=0.5, trim_x=50, trim_y=50, min_cluster_size=5), **kw})
            for i, (m, kw, _) in enumerate(scenes)]
    pts = [p for _, _, p in scenes]
    maxp = max(len(p) for p in pts)
    want = []
    for cfg, p in zip(cfgs, pts):
        h = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=maxp)
        h.push_raw_cloud_and_pose(p, IDENTITY_POSE)
        want.append((h.tap("ground_voxels").copy(), h.tap("point_class").copy(), h.filter_cloud().copy()))

    # pipelined streaming: three frames of the scene in flight
    for (vw, cw, ow), cfg, p in zip(want, cfgs, pts):
        h = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=maxp)
        h.set_pipelining(True)
        outs = [np.empty((maxp, 8), np.float32) for _ in range(3)]
        for o in outs:
            h.submit_frame(p, IDENTITY_POSE, o)
        first = h.collect_frame().copy()
        while h.frames_in_flight():
            h.collect_frame()
        assert first.tobytes() == ow.tobytes(), "pipelined output differs from the single handle"

    # batched (same config per batch) and mixed (one config per sequence)
    d_in = [_alloc(product, maxp * 16) for _ in pts]
    d_out = [_alloc(product, maxp * 32) for _ in pts]
    try:
        for s, p in enumerate(pts):
            assert product.device_upload(0, d_in[s], p.ctypes.data_as(C.c_void_p), p.nbytes) == 0
        for s, cfg in enumerate(cfgs):
            hs = [MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=maxp) for _ in range(2)]
            SequenceBatch(hs).step_device([d_in[s].value] * 2, [len(pts[s])] * 2, [IDENTITY_POSE] * 2, [d_out[s].value, d_out[1 - s].value])
            for h in hs:
                h.sync()
                assert h.tap("ground_voxels").tobytes() == want[s][0].tobytes(), "batched ground voxels"
                assert h.tap("point_class").tobytes() == want[s][1].tobytes(), "batched point classes"
        hs = [MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=maxp) for cfg in cfgs]
        MixedBatch(product).step(hs, [d.value for d in d_in], [len(p) for p in pts], [IDENTITY_POSE] * 2, [d.value for d in d_out])
        for s, h in enumerate(hs):
            h.sync()
            assert h.tap("ground_voxels").tobytes() == want[s][0].tobytes(), "mixed ground voxels"
            assert h.tap("point_class").tobytes() == want[s][1].tobytes(), "mixed point classes"
    finally:
        for d in d_in + d_out:
            product.device_free(0, d)
