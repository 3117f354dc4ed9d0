"""GPU parity on the edge cases the oracle tests cover: empty / tiny / non-finite inputs, arbitrary
point_step and field offsets, missing intensity, min_cluster_size 1, the ExtractIndices overflow quirk,
push-push-filter call patterns, and a randomised property test of cluster membership."""
import numpy as np
import pytest

from dynamicslamtool_b200 import MovingObjectRemoval
from dynamicslamtool_b200.binding import NO_FIELD
from helpers import IDENTITY_POSE, OPEN_CFG, blob, components_min_label, f32_sqdist_matrix, with_intensity, write_cfg
from parity import ParityStats, compare_frame

pytestmark = pytest.mark.gpu


def pair(product, oracle, cfg, **kw):
    return MovingObjectRemoval(cfg, 4, 3, binding=product, **kw), MovingObjectRemoval(cfg, 4, 3, binding=oracle)


def step(gpu, orc, pts, pose=IDENTITY_POSE, **kw):
    gpu.push_raw_cloud_and_pose(pts, pose, **kw)
    orc.push_raw_cloud_and_pose(pts, pose, **kw)
    og, oo = gpu.filter_cloud().copy(), orc.filter_cloud().copy()
    bad = compare_frame(gpu, orc, og, oo)
    assert not bad, bad
    return og


def test_empty_tiny_and_nonfinite(product, oracle, tmp_path):
    gpu, orc = pair(product, oracle, write_cfg(tmp_path))
    step(gpu, orc, np.zeros((0, 4), np.float32))
    step(gpu, orc, np.zeros((1, 4), np.float32))
    pts = np.array([[0, 0, 0, 1], [3.0, 0, 0, 1], [3.0000002, 0, 0, 1], [-3.0, -3.0, -0.5, 1], [0, 0, -0.50000006, 1], [0, 0, 5.0, 1],
                    [0, 0, 5.000001, 1], [np.nan, 0, 0, 1], [0, np.inf, 0, 1], [0, 0, -np.inf, 1], [0, -3.1, 0, 1]], np.float32)
    out = step(gpu, orc, pts)
    assert out.shape == (6, 8)
    step(gpu, orc, np.zeros((0, 4), np.float32))


def test_point_step_and_offsets(product, oracle, tmp_path):
    rng = np.random.default_rng(0)
    gpu, orc = pair(product, oracle, write_cfg(tmp_path, ec_distance_threshold=0.3, min_cluster_size=20, max_cluster_size=5000, **OPEN_CFG))
    xyz = np.concatenate([blob(rng, (0, 0, 0), 300, 0.1), blob(rng, (3, 1, 0), 200, 0.1)])
    # Velodyne-style record: x y z pad intensity ring(u16) pad time -> 32 B, intensity at 16 (PCL PointXYZI layout)
    rec = np.zeros((len(xyz), 8), np.float32)
    rec[:, :3] = xyz
    rec[:, 4] = rng.uniform(0, 1, len(xyz))
    rec[:, 5:] = 123.0
    blob32 = rec.view(np.uint8).reshape(-1)
    for f in range(3):
        step(gpu, orc, blob32, point_step=32, offsets=(0, 4, 8, 16))
    # 12-byte xyz-only points, no intensity field
    gpu, orc = pair(product, oracle, write_cfg(tmp_path, ec_distance_threshold=0.3, min_cluster_size=20, max_cluster_size=5000, **OPEN_CFG))
    out = step(gpu, orc, np.ascontiguousarray(xyz))
    assert np.all(out[:, 4] == 0.0)
    # fields in a scrambled order: z, intensity, y, x at 20 B
    rec = np.stack([xyz[:, 2], np.full(len(xyz), 0.25, np.float32), xyz[:, 1], xyz[:, 0], np.zeros(len(xyz), np.float32)], axis=1).astype(np.float32)
    step(gpu, orc, np.ascontiguousarray(rec).view(np.uint8).reshape(-1), point_step=20, offsets=(12, 8, 0, 4))


@pytest.mark.parametrize("seed", range(6))
def test_membership_property_random_clouds(product, oracle, tmp_path, seed):
    rng = np.random.default_rng(100 + seed)
    r = float(rng.choice([0.05, 0.11, 0.3, 0.7]))
    n = int(rng.integers(500, 3000))
    xyz = np.concatenate([rng.uniform(-3, 3, (n, 3)), *(blob(rng, rng.uniform(-3, 3, 3), n // 8, r * 0.6) for _ in range(6))]).astype(np.float32)
    # duplicates and points exactly on cell boundaries / at the radius
    xyz = np.concatenate([xyz, xyz[:50], xyz[:50] + np.float32([r, 0, 0])]).astype(np.float32)
    cfg = write_cfg(tmp_path, ec_distance_threshold=r, min_cluster_size=1, max_cluster_size=100000, **OPEN_CFG)
    gpu = MovingObjectRemoval(cfg, 4, 3, binding=product, max_clusters=16384)
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    step(gpu, orc, with_intensity(xyz))
    r2 = np.float32(np.float64(np.float32(r)) * np.float64(np.float32(r)))
    want = components_min_label(f32_sqdist_matrix(xyz) < r2)  # independent of both implementations
    np.testing.assert_array_equal(gpu.tap("labels"), want)
    # permutation invariance of the partition
    perm = rng.permutation(len(xyz))
    step(gpu, orc, with_intensity(xyz[perm]))
    lab = gpu.tap("labels")
    inv = np.empty_like(perm)
    inv[perm] = np.arange(len(perm))
    a, b = want, lab[inv]
    assert len(set(zip(a.tolist(), b.tolist()))) == len(set(a.tolist())) == len(set(b.tolist()))


def test_extract_overflow_and_tracker_timeline(product, oracle, tmp_path):
    rng = np.random.default_rng(11)
    gpu, orc = pair(product, oracle, write_cfg(tmp_path, ec_distance_threshold=0.3, min_cluster_size=50, max_cluster_size=5000, **OPEN_CFG))
    base = blob(rng, (0, 0, 0), 300, 0.1)
    seen = False
    for f in range(12):
        out = step(gpu, orc, with_intensity(base + np.float32([0.45 * f, 0, 0])))
        seen |= bool(gpu.counts()["EXTRACT_OVERFLOW"])
    assert seen


def test_push_push_filter_and_double_filter(product, oracle, tmp_path):
    rng = np.random.default_rng(12)
    gpu, orc = pair(product, oracle, write_cfg(tmp_path, ec_distance_threshold=0.3, min_cluster_size=50, max_cluster_size=5000, **OPEN_CFG))
    a, b = blob(rng, (2, 0, 0), 300, 0.12), blob(rng, (-2, 1, 0), 300, 0.12)
    for f in range(8):
        pts = with_intensity(np.concatenate([a, b + np.float32([0.12 * f, 0, 0])]))
        if f % 3 == 1:  # push without filter
            gpu.push_raw_cloud_and_pose(pts, IDENTITY_POSE)
            orc.push_raw_cloud_and_pose(pts, IDENTITY_POSE)
            assert not compare_frame(gpu, orc, None, None, after_filter=False)
            continue
        step(gpu, orc, pts)
        if f % 3 == 2:  # filter twice
            og, oo = gpu.filter_cloud().copy(), orc.filter_cloud().copy()
            assert not compare_frame(gpu, orc, og, oo)


def test_capacity_errors_are_reported(product, tmp_path):
    from dynamicslamtool_b200 import MorError
    gpu = MovingObjectRemoval(write_cfg(tmp_path), 4, 3, binding=product, max_points=1000)
    lim = gpu.limits
    assert (lim.max_points, lim.max_clusters, lim.max_moving) == (1000, 8192, 1024) and lim.max_cells >= 1 << 24
    with pytest.raises(MorError) as e:
        gpu.push_raw_cloud_and_pose(np.zeros((1001, 4), np.float32), IDENTITY_POSE)
    assert e.value.status == 6
    with pytest.raises(MorError):
        MovingObjectRemoval(tmp_path / "missing.txt", 4, 3, binding=product)


def test_device_resident_api_matches_host_api(product, tmp_path):
    import ctypes as C
    rng = np.random.default_rng(13)
    cfg = write_cfg(tmp_path, ec_distance_threshold=0.3, min_cluster_size=50, max_cluster_size=5000, **OPEN_CFG)
    host, dev = MovingObjectRemoval(cfg, 4, 3, binding=product), MovingObjectRemoval(cfg, 4, 3, binding=product)
    a, b = blob(rng, (2, 0, 0), 300, 0.12), blob(rng, (-2, 1, 0), 300, 0.12)
    d_in, d_out = C.c_void_p(), C.c_void_p()
    assert product.device_alloc(0, 600 * 16, C.byref(d_in)) == 0 and product.device_alloc(0, 600 * 32, C.byref(d_out)) == 0
    for f in range(7):
        pts = with_intensity(np.concatenate([a, b + np.float32([0.12 * f, 0, 0])]))
        host.push_raw_cloud_and_pose(pts, IDENTITY_POSE)
        want = host.filter_cloud().copy()
        assert product.device_upload(0, d_in, pts.ctypes.data_as(C.c_void_p), pts.nbytes) == 0
        dev.push_device(d_in.value, 600, IDENTITY_POSE)
        n = dev.filter_device(d_out.value, 600)
        got = np.empty((n, 8), np.float32)
        assert product.device_download(0, got.ctypes.data_as(C.c_void_p), d_out, n * 32) == 0
        np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))
    product.device_free(0, d_in)
    product.device_free(0, d_out)


def test_batched_step_matches_oracle_per_sequence(product, oracle, cfg_dir):
    """mor_batch_step_device: S sequences advanced by one set of launches give, per sequence, exactly what the
    oracle gives for that sequence alone (independence of the replicas, SURVEY §8e / BASELINE config 5)."""
    import ctypes as C
    from dynamicslamtool_b200 import SequenceBatch, Synth
    cfg = cfg_dir / "MOR_config.txt"
    S, frames = 3, 8
    syn = [Synth(1, 40 + s) for s in range(S)]
    maxp = syn[0].max_points
    gpus = [MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=maxp) for _ in range(S)]
    orcs = [MovingObjectRemoval(cfg, 4, 3, binding=oracle) for _ in range(S)]
    batch = SequenceBatch(gpus)
    d_in, d_out = [], []
    for s in range(S):
        a, b = C.c_void_p(), C.c_void_p()
        assert product.device_alloc(0, maxp * 16, C.byref(a)) == 0 and product.device_alloc(0, maxp * 32, C.byref(b)) == 0
        d_in.append(a); d_out.append(b)
    for f in range(frames):
        data = [syn[s].frame(f) for s in range(S)]
        for s in range(S):
            pts = data[s][0]
            assert product.device_upload(0, d_in[s], pts.ctypes.data_as(C.c_void_p), pts.nbytes) == 0
        batch.step_device([p.value for p in d_in], [d[0].shape[0] for d in data], [d[1] for d in data], [p.value for p in d_out])
        for s in range(S):
            orcs[s].push_raw_cloud_and_pose(*data[s])
            oo = orcs[s].filter_cloud().copy()
            gpus[s].sync()
            n_out = gpus[s].counts()["NOUT"]
            og = np.empty((n_out, 8), np.float32)
            if n_out:
                assert product.device_download(0, og.ctypes.data_as(C.c_void_p), d_out[s], n_out * 32) == 0
            bad = compare_frame(gpus[s], orcs[s], og, oo)
            assert not bad, f"sequence {s} frame {f}: {bad}"
    # batched handles (the leader and a follower) can go back to single stepping, and back into a batch
    for s in (0, 2):
        pts, pose = syn[s].frame(frames)
        gpus[s].push_raw_cloud_and_pose(pts, pose); orcs[s].push_raw_cloud_and_pose(pts, pose)
        og, oo = gpus[s].filter_cloud().copy(), orcs[s].filter_cloud().copy()
        assert not compare_frame(gpus[s], orcs[s], og, oo)
    pts1, pose1 = syn[1].frame(frames)
    gpus[1].push_raw_cloud_and_pose(pts1, pose1); orcs[1].push_raw_cloud_and_pose(pts1, pose1)
    gpus[1].filter_cloud(); orcs[1].filter_cloud()
    data = [syn[s].frame(frames + 1) for s in range(S)]
    for s in range(S):
        assert product.device_upload(0, d_in[s], data[s][0].ctypes.data_as(C.c_void_p), data[s][0].nbytes) == 0
    batch.step_device([p.value for p in d_in], [d[0].shape[0] for d in data], [d[1] for d in data], [p.value for p in d_out])
    for s in range(S):
        orcs[s].push_raw_cloud_and_pose(*data[s])
        oo = orcs[s].filter_cloud().copy()
        gpus[s].sync()
        n_out = gpus[s].counts()["NOUT"]
        og = np.empty((n_out, 8), np.float32)
        assert product.device_download(0, og.ctypes.data_as(C.c_void_p), d_out[s], n_out * 32) == 0
        assert not compare_frame(gpus[s], orcs[s], og, oo)
    for p in d_in + d_out:
        product.device_free(0, p)


def test_refused_batched_step_launches_nothing(product, oracle, cfg_dir):
    """A lockstep batched step that a later sequence's frame refuses (n > max_points) launches nothing, not even the
    pending back half of an earlier, pipelined sequence; the step after it equals the oracle in every sequence."""
    import ctypes as C
    from dynamicslamtool_b200 import MorError, SequenceBatch, Synth
    cfg = cfg_dir / "MOR_config.txt"
    S = 3
    syn = [Synth(1, 50 + s) for s in range(S)]
    maxp = syn[0].max_points
    gpus = [MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=maxp) for _ in range(S)]
    orcs = [MovingObjectRemoval(cfg, 4, 3, binding=oracle) for _ in range(S)]
    gpus[0].set_pipelining(True)
    d_in, d_out = [], []
    for s in range(S):
        a, b = C.c_void_p(), C.c_void_p()
        assert product.device_alloc(0, (maxp + 1) * 16, C.byref(a)) == 0 and product.device_alloc(0, maxp * 32, C.byref(b)) == 0
        d_in.append(a); d_out.append(b)
    try:
        for s in range(S):  # frame 0 alone; sequence 0's back half stays pending (pipelined push, filter that asks for nothing)
            pts, pose = syn[s].frame(0)
            assert product.device_upload(0, d_in[s], pts.ctypes.data_as(C.c_void_p), pts.nbytes) == 0
            gpus[s].push_device(d_in[s].value, len(pts), pose)
            if s == 0:
                gpus[s].filter_device(None, 0, want_count=False)
            else:
                gpus[s].filter_device(d_out[s].value, maxp)
            orcs[s].push_raw_cloud_and_pose(pts, pose)
            orcs[s].filter_cloud()
        data = [syn[s].frame(1) for s in range(S)]
        big = np.zeros((maxp + 1, 4), np.float32)
        big[: len(data[2][0])] = data[2][0]
        assert product.device_upload(0, d_in[2], big.ctypes.data_as(C.c_void_p), big.nbytes) == 0
        launches = [g.launch_count() for g in gpus]
        with pytest.raises(MorError) as e:
            SequenceBatch(gpus).step_device([p.value for p in d_in], [len(data[0][0]), len(data[1][0]), maxp + 1],
                                            [d[1] for d in data], [p.value for p in d_out])
        assert e.value.status == 6
        assert [g.launch_count() for g in gpus] == launches
        for s in range(S):
            pts = data[s][0]
            assert product.device_upload(0, d_in[s], pts.ctypes.data_as(C.c_void_p), pts.nbytes) == 0
        SequenceBatch(gpus).step_device([p.value for p in d_in], [len(d[0]) for d in data], [d[1] for d in data], [p.value for p in d_out])
        for s in range(S):
            orcs[s].push_raw_cloud_and_pose(*data[s])
            oo = orcs[s].filter_cloud().copy()
            gpus[s].sync()
            n_out = gpus[s].counts()["NOUT"]
            og = np.empty((n_out, 8), np.float32)
            if n_out:
                assert product.device_download(0, og.ctypes.data_as(C.c_void_p), d_out[s], n_out * 32) == 0
            bad = compare_frame(gpus[s], orcs[s], og, oo)
            assert not bad, f"sequence {s}: {bad}"
    finally:
        for p in d_in + d_out:
            product.device_free(0, p)


@pytest.mark.parametrize("n_bad,n_good", [(1, 0), (2, 1), (3, 5), (6, 2)])
def test_confidence_parameters(product, oracle, tmp_path, n_bad, n_good):
    """moving_confidence / static_confidence other than the node's 4, 3 (external_sync_test.cpp:37): ring-buffer depth,
    confirmation frame and confidence caps must follow the reference for every combination."""
    rng = np.random.default_rng(20 + n_bad)
    cfg = write_cfg(tmp_path, ec_distance_threshold=0.3, min_cluster_size=50, max_cluster_size=5000, **OPEN_CFG)
    gpu = MovingObjectRemoval(cfg, n_bad, n_good, binding=product)
    orc = MovingObjectRemoval(cfg, n_bad, n_good, binding=oracle)
    a, b, c = blob(rng, (2, 0, 0), 300, 0.12), blob(rng, (-2, 1, 0), 300, 0.12), blob(rng, (0, -3, 0.5), 250, 0.1)
    confirmed_at = None
    for f in range(14):
        move = np.float32([0.12 * min(f, 8), 0, 0])  # the mover stops after frame 8: decay path
        pts = with_intensity(np.concatenate([a, b + move, c + np.float32([0, 0.1 * f, 0])]))
        step(gpu, orc, pts)
        if confirmed_at is None and gpu.counts()["NMO"]:
            confirmed_at = f
    assert confirmed_at is not None  # the mover was confirmed for every (n_bad, n_good); parity is checked frame by frame in step()


def test_many_movers_exceed_one_block(product, oracle, tmp_path):
    """More confirmed movers than threads in a block (256) and more clusters than a warp: exercises the chunked,
    order-preserving paths of the chain / tracking code."""
    rng = np.random.default_rng(31)
    cfg = write_cfg(tmp_path, ec_distance_threshold=0.2, min_cluster_size=10, max_cluster_size=5000, opc_normalization_factor=20,
                    leave_off_distance=0.5, **OPEN_CFG)
    gpu = MovingObjectRemoval(cfg, 4, 3, binding=product, max_clusters=4096, max_moving=2048)
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    centers = np.array([[2.0 * i, 2.0 * j, 0.0] for i in range(20) for j in range(16)], np.float32)  # 320 blobs, 2 m apart
    blobs = [blob(rng, c, 24, 0.03) for c in centers]
    n_mo = []
    for f in range(8):
        pts = with_intensity(np.concatenate([bl + np.float32([0.13 * f, 0, 0]) for bl in blobs]) + rng.normal(0, 0.001, (320 * 24, 3)).astype(np.float32))
        step(gpu, orc, pts)
        n_mo.append(gpu.counts()["NMO"])
    assert max(n_mo) > 256, n_mo


def test_reset_starts_a_new_sequence(product, oracle, cfg_dir):
    """mor_reset = destroy + construct without re-allocating: after it the handle behaves exactly like a new one
    (no previous frame, empty buffers, nothing tracked), also in the middle of tracking and after a pushed frame
    that was never filtered."""
    from dynamicslamtool_b200 import Synth
    from helpers import crc
    cfg = cfg_dir / "MOR_config.txt"
    s1, s2 = Synth(1, 1), Synth(1, 5)
    gpu = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=s1.max_points)
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    for f in range(9):  # long enough for confirmed moving objects
        pts, pose = s1.frame(f)
        step(gpu, orc, pts, pose)
    assert gpu.counts()["NMO"] > 0
    pts, pose = s1.frame(9)
    gpu.push_raw_cloud_and_pose(pts, pose)  # pushed, not filtered
    gpu.reset(); orc.reset()
    fresh = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=s1.max_points)
    for f in range(8):
        pts, pose = s2.frame(f)
        fresh.push_raw_cloud_and_pose(pts, pose)
        of = fresh.filter_cloud().copy()
        og = step(gpu, orc, pts, pose)
        assert crc(og) == crc(of)
        for t in ("labels", "cluster_id", "centroids", "match_score", "flags", "mo_centroids", "mo_conf", "removed_mask"):
            assert crc(gpu.tap(t)) == crc(fresh.tap(t)), t


def test_visualize_outputs_cluster_collection_and_markers(product, oracle, cfg_dir):
    """The reference's VISUALIZE side outputs: cluster_collection (cpp:226-229, :553-558) byte for byte - a stable
    partition of the cloud by cluster - and one marker per mo_vec entry (cpp:640-642): cluster, id, colour and
    bounding-box scale exact, position = centroid (the reference accumulates it in float: 1e-5 relative)."""
    from dynamicslamtool_b200 import Synth
    for scen, cfg, frames in ((1, "MOR_config.txt", range(0, 12)), (2, "MOR_config_hdl64.txt", range(100, 108))):
        s = Synth(scen, scen)
        gpu = MovingObjectRemoval(cfg_dir / cfg, 4, 3, binding=product, max_points=s.max_points)
        orc = MovingObjectRemoval(cfg_dir / cfg, 4, 3, binding=oracle)
        seen_markers = 0
        for f in frames:
            pts, pose = s.frame(f)
            gpu.push_raw_cloud_and_pose(pts, pose); orc.push_raw_cloud_and_pose(pts, pose)
            cg, co = gpu.cluster_collection(), orc.cluster_collection()   # between push and filter, as the reference publishes it
            assert cg.shape == co.shape and cg.tobytes() == co.tobytes(), f"scenario {scen} frame {f}"
            assert cg.shape[0] == gpu.counts()["NK"]
            og, oo = gpu.filter_cloud().copy(), orc.filter_cloud().copy()
            assert og.tobytes() == oo.tobytes()
            assert gpu.cluster_collection().tobytes() == co.tobytes()       # and after filter: same frame, same answer
            mg, mo = gpu.moving_markers(), orc.moving_markers()
            assert mg.shape == mo.shape
            seen_markers += mg.shape[0]
            for name in ("cluster", "id", "color", "scale"):
                assert np.array_equal(mg[name], mo[name]), name
            # filterCloud's marker counter starts at 1 and advances once per looked-up entry (reference cpp:622, :669)
            assert np.array_equal(mg["id"], np.arange(1, mg.shape[0] + 1)), mg["id"]
            np.testing.assert_allclose(mg["position"], mo["position"], rtol=1e-5, atol=1e-5)
        assert seen_markers > 0


def test_run_to_run_determinism(product, cfg_dir):
    """Intra-cell order, union order and atomic order vary from run to run; every observable (labels, cluster order,
    centroids bit for bit, scores, flags, mo_vec, masks, output bytes) must not."""
    from dynamicslamtool_b200 import Synth
    from helpers import crc
    cfg = cfg_dir / "MOR_config_hdl64.txt"
    s = Synth(2, 2)
    frames = [s.frame(f) for f in range(100, 108)]  # the dense stretch: cells with > 1000 points, 27k-point clusters

    def run():
        m = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=s.max_points)
        sig = []
        for pts, pose in frames:
            m.push_raw_cloud_and_pose(pts, pose)
            out = m.filter_cloud()
            sig.append(tuple(crc(m.tap(t)) for t in ("labels", "cluster_id", "cluster_root", "cluster_size", "centroids", "cluster_bbox", "match_query",
                                                       "match_match", "match_score", "flags", "mo_centroids", "mo_conf", "removed_mask")) + (crc(out),))
        return sig

    a, b, c = run(), run(), run()
    assert a == b == c


@pytest.mark.parametrize("r", [0.11, 0.03])
def test_small_radius_over_a_large_crop_box(product, oracle, cfg_dir, tmp_path, r):
    """Outdoor trim with the indoor clustering radius (and a quarter of it): 80 m x 80 m x 4.4 m at r = 0.11 m is
    1.1e8 cells of edge r/sqrt(3), at r = 0.03 m 5e9. The clustering grid is a hash table of the occupied cells, so
    neither the crop box nor the radius bounds anything: no capacity error exists on this path."""
    from dynamicslamtool_b200 import Synth
    cfg = write_cfg(tmp_path, base=cfg_dir / "MOR_config_hdl64.txt", ec_distance_threshold=r, min_cluster_size=20 if r > 0.1 else 3)
    s = Synth(2, 2)
    gpu = MovingObjectRemoval(cfg, 4, 3, binding=product, max_points=s.max_points)
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    for f in range(3):
        step(gpu, orc, *s.frame(f))


def test_trimming_disabled_with_huge_limits(product, oracle, tmp_path):
    """trim_* = 1e6 m ("disabled"): the grid follows no box at all. Points kilometres apart still cluster exactly."""
    rng = np.random.default_rng(77)
    cfg = write_cfg(tmp_path, trim_x=1e6, trim_y=1e6, trim_z=1e6, gp_limit=-1e6, ec_distance_threshold=0.3, min_cluster_size=50, max_cluster_size=5000)
    gpu = MovingObjectRemoval(cfg, 4, 3, binding=product)
    orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
    far = [blob(rng, c, 200, 0.1) for c in ((0, 0, 0), (3000, -2500, 40), (-9000.5, 8000.25, -3), (20000, 20000, 100))]
    for f in range(6):
        pts = with_intensity(np.concatenate([b + np.float32([0.12 * f * (i % 2), 0, 0]) for i, b in enumerate(far)]))
        step(gpu, orc, pts)
    assert gpu.counts()["K"] == 4


def test_unaligned_point_step(product, oracle, tmp_path):
    """pcl::fromPCLPointCloud2 maps fields by name whatever the record layout (cpp:523): the 22-byte XYZIRT record of
    the stock velodyne driver (x@0 y@4 z@8 intensity@12 ring@16 time@18) has no 4-byte alignment from the second
    point on; a packed 13-byte record with odd offsets even less."""
    rng = np.random.default_rng(5)
    cfg = write_cfg(tmp_path, ec_distance_threshold=0.3, min_cluster_size=50, max_cluster_size=5000, **OPEN_CFG)
    for step_b, offs in ((22, (0, 4, 8, 12)), (13, (1, 5, 9, NO_FIELD)), (19, (3, 7, 11, 15))):
        gpu = MovingObjectRemoval(cfg, 4, 3, binding=product)
        orc = MovingObjectRemoval(cfg, 4, 3, binding=oracle)
        ref = MovingObjectRemoval(cfg, 4, 3, binding=product)
        a, b = blob(rng, (2, 0, 0), 300, 0.12), blob(rng, (-2, 1, 0), 300, 0.12)
        for f in range(7):
            pts = with_intensity(np.concatenate([a, b + np.float32([0.12 * f, 0, 0])]), 0.25)
            rec = np.full((len(pts), step_b), 0xA5, np.uint8)
            for col, off in enumerate(offs):
                if off != NO_FIELD:
                    rec[:, off:off + 4] = pts[:, col:col + 1].copy().view(np.uint8)
            rec = np.ascontiguousarray(rec)
            gpu.push_raw_cloud_and_pose(rec, IDENTITY_POSE, point_step=step_b, offsets=offs)
            orc.push_raw_cloud_and_pose(rec, IDENTITY_POSE, point_step=step_b, offsets=offs)
            og, oo = gpu.filter_cloud().copy(), orc.filter_cloud().copy()
            assert not compare_frame(gpu, orc, og, oo)
            plain = pts if offs[3] != NO_FIELD else np.ascontiguousarray(pts[:, :3])
            ref.push_raw_cloud_and_pose(plain, IDENTITY_POSE)
            assert ref.filter_cloud().tobytes() == og.tobytes()


@pytest.mark.parametrize("seed", range(18))
def test_fuzz_random_configs_and_scenes(product, oracle, tmp_path, seed):
    """Randomised end-to-end parity: random crop box, radius, cluster size limits, method, thresholds and confidence
    counts over a random scene of static / moving / appearing / vanishing blobs, a plane of ground points, NaNs and
    out-of-range points, with a random rigid motion of the sensor between frames."""
    from scipy.spatial.transform import Rotation as R
    rng = np.random.default_rng(1000 + seed)
    r = float(rng.choice([0.08, 0.15, 0.3, 0.6]))
    cfgkw = dict(
        trim_x=float(rng.uniform(4, 9)), trim_y=float(rng.uniform(4, 9)), trim_z=float(rng.uniform(1.5, 4)), gp_limit=float(rng.uniform(-1.2, -0.4)),
        ec_distance_threshold=r, min_cluster_size=int(rng.integers(5, 60)), max_cluster_size=int(rng.integers(400, 3000)),
        method_choice=int(rng.integers(1, 3)), opc_normalization_factor=int(rng.integers(2, 25)), volume_constraint=float(rng.uniform(0.1, 0.6)),
        pde_lb=float(rng.uniform(0.001, 0.01)), pde_ub=float(rng.uniform(0.2, 0.8)), pde_distance_threshold=float(rng.uniform(0.05, 0.4)),
        leave_off_distance=float(rng.uniform(0.2, 1.0)), catch_up_distance=float(rng.uniform(0.1, 0.6)))
    if seed >= 12:  # the voxel-covariance ground modes (reference cpp:90-200) instead of the crop
        cfgkw.update(ground_mode=1 + seed % 2, gp_leaf=float(rng.choice([0.2, 0.35, 0.5])), gp_bin_width=float(rng.choice([0.2, 0.5])),
                     gp_planarity=float(rng.choice([0.005, 0.02])))
    cfg = write_cfg(tmp_path, **cfgkw)
    n_bad, n_good = int(rng.integers(1, 6)), int(rng.integers(0, 5))
    gpu = MovingObjectRemoval(cfg, n_bad, n_good, binding=product)
    orc = MovingObjectRemoval(cfg, n_bad, n_good, binding=oracle)
    nb = int(rng.integers(4, 14))
    centers = rng.uniform(-6, 6, (nb, 3)) * np.array([1, 1, 0.15])
    vel = rng.uniform(-0.25, 0.25, (nb, 3)) * np.array([1, 1, 0]) * (rng.random((nb, 1)) < 0.5)
    sizes = rng.integers(30, 900, nb)
    sig = rng.uniform(0.5, 1.5, nb) * r
    shapes = [rng.normal(0, 1, (int(sizes[b]), 3)) * sig[b] * np.array([1, 1, 0.6]) for b in range(nb)]
    ground = np.concatenate([rng.uniform(-9, 9, (3000, 2)), rng.normal(-1.5, 0.02, (3000, 1))], axis=1)
    pos, yaw = np.zeros(3), 0.0
    for f in range(12):
        pos = pos + rng.uniform(-0.15, 0.15, 3) * np.array([1, 1, 0.1])
        yaw += float(rng.uniform(-0.05, 0.05))
        rot = R.from_euler("zyx", [yaw, float(rng.uniform(-0.01, 0.01)), float(rng.uniform(-0.01, 0.01))])
        world = [shapes[b] + centers[b] + vel[b] * f + rng.normal(0, 0.003, shapes[b].shape) for b in range(nb) if not (b % 5 == 4 and f % 6 >= 4)]
        world.append(ground + rng.normal(0, 0.002, ground.shape))
        w = np.concatenate(world)
        sensor = rot.inv().apply(w - pos).astype(np.float32)  # world -> sensor frame, consistent with the odometry pose
        pts = with_intensity(sensor, 0.3)
        pts[rng.integers(0, len(pts), 5), rng.integers(0, 3, 5)] = np.nan
        pts[rng.integers(0, len(pts), 3), 0] = np.inf
        pose = np.concatenate([pos, rot.as_quat()])
        step(gpu, orc, np.ascontiguousarray(pts), pose)


def test_radius_tie_counter_equals_the_oracles(product, oracle, cfg_dir):
    """mor_count_radius_ties (north_star: divergence at the exact radius counted): the same brute-force count on both sides,
    on real frames (C1, 29k points; the first frames of C2) and for several band widths."""
    from dynamicslamtool_b200 import Synth
    for scenario, cfg, frames in ((1, "MOR_config.txt", 3), (2, "MOR_config_hdl64.txt", 2)):
        s = Synth(scenario, scenario)
        gpu = MovingObjectRemoval(cfg_dir / cfg, 4, 3, binding=product, max_points=s.max_points)
        orc = MovingObjectRemoval(cfg_dir / cfg, 4, 3, binding=oracle)
        for f in range(frames):
            pts, pose = s.frame(f)
            gpu.push_raw_cloud_and_pose(pts, pose); orc.push_raw_cloud_and_pose(pts, pose)
            for ulps in (0, 2, 64):
                assert gpu.radius_ties(ulps) == orc.radius_ties(ulps), (scenario, f, ulps)
            gpu.filter_cloud(); orc.filter_cloud()
        assert orc.radius_ties(1 << 12) > 0  # a band wide enough to hold pairs: the counters do count
