"""CPU-only checks of the checker itself: the restatement against the golden vectors recorded from the compiled
reference (tests/golden/make_golden.py), and its pieces against independent numpy answers."""
import hashlib
import math
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def _golden(name):
    return np.load(os.path.join(HERE, "golden", name))


def _sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def assert_input(a, g, key):
    """The generator reproduced the input the golden run was recorded on."""
    assert _sha256(a) == str(g[key + "__sha256"]), f"{key}: synth no longer generates the recorded input"


def assert_golden(got, g, key):
    """Bit-exact comparison with a recorded array, stored whole or as SHA-256 + shape + evenly spaced sample rows."""
    if key in g.files:
        np.testing.assert_array_equal(got, g[key], err_msg=key)
        return
    got = np.ascontiguousarray(got)
    assert got.shape == tuple(g[key + "__shape"]), (key, got.shape, tuple(g[key + "__shape"]))
    rows = np.unique(np.linspace(0, got.shape[0] - 1, 16).astype(np.int64))
    np.testing.assert_array_equal(got[rows], g[key + "__sample"], err_msg=key)
    assert _sha256(got) == str(g[key + "__sha256"]), key


@pytest.fixture(scope="module")
def golden_pipe():
    return np.load(os.path.join(HERE, "golden", "pipeline_vlp16_600.npz"))


@pytest.fixture(scope="module")
def golden_pieces():
    return np.load(os.path.join(HERE, "golden", "pieces.npz"))


def test_restatement_reproduces_golden_pipeline(oracle, golden_pipe):
    g = golden_pipe
    pipe = oracle.pipeline()
    pipe.seed_map(g["map_corner"], g["map_surf"])
    for i in range(6):
        ok, odom, aft, _ = pipe.sweep(g[f"pts{i}"], g[f"rings{i}"])
        assert ok
        # the restatement shares the shim's dense algebra with the recorded reference build: bit-exact
        np.testing.assert_array_equal(odom, g[f"odom{i}"])
        np.testing.assert_array_equal(aft, g[f"aft{i}"])
        if i in (0, 3):
            for name in ("sharp", "less_sharp", "flat", "less_flat"):
                np.testing.assert_array_equal(pipe.scanreg.cloud(name), g[f"{name}{i}"])
    np.testing.assert_array_equal(pipe.mapping.cloud("corner_cubes"), g["final_corner_cubes"])
    assert pipe.mapping.cloud("surf_cubes").shape[0] == int(g["final_surf_cubes_n"][0])


def test_restatement_pieces_match_golden(oracle, golden_pieces):
    g = golden_pieces
    idx5, d5 = oracle.knn(g["knn_pts"], g["knn_q"], 5)
    np.testing.assert_array_equal(d5, g["knn_d5"])
    np.testing.assert_array_equal(idx5, g["knn_idx5"])
    idx1, d1 = oracle.knn(g["knn_corner"], g["knn_q"], 1)
    np.testing.assert_array_equal(idx1, g["knn_idx1"])
    np.testing.assert_array_equal(d1, g["knn_d1"])
    np.testing.assert_array_equal(oracle.voxel_grid(g["vox_in"], 0.4), g["vox_out"])
    np.testing.assert_array_equal(oracle.qr_solve6(g["A"], g["b"]), g["x"])
    ev, V = oracle.eig_sym(g["A"])
    np.testing.assert_array_equal(ev, g["ev"])
    np.testing.assert_array_equal(V, g["V"])
    np.testing.assert_array_equal(oracle.lsq53(g["P5"]), g["x53"])


def test_restatement_equals_compiled_reference_live(oracle, scene):
    """Full pipeline, bit for bit, against the compiled reference's run on a second trajectory (60 k map, VLP-16 at 900
    azimuth steps, backwards yaw, sideways drift) recorded in golden/pipeline_vlp16_900_live.npz."""
    from loam_velodyne_b200 import synth
    g = _golden("pipeline_vlp16_900_live.npz")
    lidar = synth.Lidar(16, 900, -15.0, 15.0)
    corner, surf = synth.make_map(scene, 60_000)
    assert_input(corner, g, "map_corner")
    assert_input(surf, g, "map_surf")
    po = oracle.pipeline()
    po.seed_map(corner, surf)
    for i in range(5):
        pts, rs = synth.make_sweep(scene, lidar, 20 + i, yaw_rate=math.radians(-7.0), v=(0.3, 0.0, 1.5))
        assert_input(pts, g, f"pts{i}")
        ok_o, od_o, aft_o, _ = po.sweep(pts, rs)
        assert ok_o == bool(g[f"ok{i}"])
        np.testing.assert_array_equal(od_o, g[f"odom{i}"])
        np.testing.assert_array_equal(aft_o, g[f"aft{i}"])
        for name in ("sharp", "less_sharp", "flat", "less_flat"):
            assert_golden(po.scanreg.cloud(name), g, f"{name}{i}")
        for name in ("last_corner", "last_surf"):
            assert_golden(po.odom.cloud(name), g, f"{name}{i}")


VARIANTS = {
    # name: (rings, azimuth steps, lower, upper, yaw rate deg/s, velocity, max range, registration overrides, odom / map iterations)
    "hdl32_ragged": (32, 700, -30.67, 10.67, 12.0, (0.5, 0.0, 2.0), 35.0, {}, (25, 10)),
    "vlp16_params": (16, 900, -15.0, 15.0, -4.0, (0.0, 0.0, 0.8), 0.0,
                     dict(n_regions=4, curv_region=3, max_sharp=3, max_flat=6, less_flat_leaf=0.3, curv_thr=0.05), (25, 10)),
    "vlp16_few_iterations": (16, 600, -15.0, 15.0, 20.0, (1.0, 0.0, 4.0), 0.0, {}, (3, 2)),
    "single_region": (16, 400, -15.0, 15.0, 5.0, (0.0, 0.0, 1.0), 25.0, dict(n_regions=1, curv_region=7), (25, 10)),
}


@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_restatement_equals_compiled_reference_variants(oracle, scene, variant):
    """Other sensor geometries, ragged rings (returns beyond max range dropped), non-default RegistrationParams and tight
    iteration budgets: the restatement agrees bit for bit on poses, features and map with the compiled reference's run
    recorded in golden/pipeline_variants.npz."""
    from loam_velodyne_b200 import synth
    g = _golden("pipeline_variants.npz")
    R, A, lo, hi, yaw, v, max_range, reg, (oi, mi) = VARIANTS[variant]
    lidar = synth.Lidar(R, A, lo, hi)
    corner, surf = synth.make_map(scene, 40_000)
    assert_input(corner, g, "map_corner")
    assert_input(surf, g, "map_surf")
    po = oracle.pipeline(odom_iter=oi, map_iter=mi)
    if reg:
        po.scanreg.configure(**reg)
    po.seed_map(corner, surf)
    for i in range(4):
        pts, rs = synth.make_sweep(scene, lidar, 5 + i, yaw_rate=math.radians(yaw), v=v, max_range=max_range)
        assert_input(pts, g, f"{variant}/pts{i}")
        if max_range > 0:
            assert len(set(rs.tolist())) > 1  # the rings really are ragged
        ok_o, od_o, aft_o, _ = po.sweep(pts, rs)
        assert ok_o == bool(g[f"{variant}/ok{i}"])
        np.testing.assert_array_equal(od_o, g[f"{variant}/odom{i}"])
        np.testing.assert_array_equal(aft_o, g[f"{variant}/aft{i}"])
        for name in ("sharp", "less_sharp", "flat", "less_flat"):
            assert_golden(po.scanreg.cloud(name), g, f"{variant}/{name}{i}")
    assert_golden(po.mapping.cloud("corner_cubes"), g, f"{variant}/corner_cubes")
    assert_golden(po.mapping.cloud("surf_cubes"), g, f"{variant}/surf_cubes")


def test_knn_against_brute_force(oracle):
    rng = np.random.RandomState(0)
    pts = np.zeros((3000, 4), np.float32)
    pts[:, :3] = rng.uniform(-20, 20, (3000, 3))
    q = np.zeros((200, 4), np.float32)
    q[:, :3] = rng.uniform(-22, 22, (200, 3))
    idx, d2 = oracle.knn(pts, q, 5)
    # same float arithmetic as nanoflann's L2_Simple_Adaptor: ((dx*dx + dy*dy) + dz*dz) in fp32
    diff = q[:, None, :3] - pts[None, :, :3]
    sq = (diff * diff).astype(np.float32)
    bf = ((sq[..., 0] + sq[..., 1]).astype(np.float32) + sq[..., 2]).astype(np.float32)
    order = np.argsort(bf, axis=1, kind="stable")[:, :5]
    np.testing.assert_array_equal(d2, np.take_along_axis(bf, order, axis=1))
    np.testing.assert_array_equal(idx, order.astype(np.int32))
    assert (np.diff(d2, axis=1) >= 0).all()


def test_voxel_grid_known_answer(oracle):
    pts = np.array([[0.05, 0.05, 0.05, 1.0], [0.15, 0.05, 0.05, 3.0],   # same 0.2 voxel
                    [0.25, 0.05, 0.05, 5.0],                             # next voxel in x
                    [0.05, 0.25, 0.05, 7.0],                             # next voxel in y
                    [-0.05, 0.05, 0.05, 9.0]], np.float32)               # voxel at negative x
    out = oracle.voxel_grid(pts, 0.2)
    # ascending voxel index, x fastest: (-1,0,0), (0,0,0), (1,0,0), (0,1,0)
    expect = np.array([[-0.05, 0.05, 0.05, 9.0], [0.10, 0.05, 0.05, 2.0], [0.25, 0.05, 0.05, 5.0],
                       [0.05, 0.25, 0.05, 7.0]], np.float32)
    np.testing.assert_allclose(out, expect, rtol=0, atol=1e-6)
    assert oracle.voxel_grid(np.zeros((0, 4), np.float32), 0.2).shape == (0, 4)


def test_dense_algebra_against_numpy(oracle):
    rng = np.random.RandomState(3)
    for _ in range(20):
        M = rng.normal(size=(6, 6))
        A = (M @ M.T + np.eye(6)).astype(np.float32)
        b = rng.normal(size=6).astype(np.float32)
        x = oracle.qr_solve6(A, b)
        np.testing.assert_allclose(x, np.linalg.solve(A.astype(np.float64), b.astype(np.float64)), rtol=2e-3, atol=2e-4)
        ev, V = oracle.eig_sym(A)
        w = np.linalg.eigvalsh(A.astype(np.float64))
        np.testing.assert_allclose(ev, w, rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(A @ V, V * ev[None, :], atol=5e-4 * np.abs(w).max())
        assert (np.diff(ev) >= 0).all()
        A3 = A[:3, :3].copy()
        ev3, V3 = oracle.eig_sym(A3)
        np.testing.assert_allclose(ev3, np.linalg.eigvalsh(A3.astype(np.float64)), rtol=1e-4, atol=1e-4)
        P = (rng.normal(size=(5, 3)) + np.array([10.0, -3.0, 25.0])).astype(np.float32)
        x53 = oracle.lsq53(P)
        ref = np.linalg.lstsq(P.astype(np.float64), -np.ones(5), rcond=None)[0]
        np.testing.assert_allclose(x53, ref, rtol=5e-3, atol=5e-4)


def test_feature_edge_cases_do_not_crash(oracle):
    """Empty rings, rings at the skip limit (<= 2*curvatureRegion + 1 points), a single huge region."""
    rng = np.random.RandomState(1)
    sizes = np.array([0, 11, 12, 0, 300, 5, 0], np.int32)
    n = int(sizes.sum())
    pts = np.zeros((n, 4), np.float32)
    ang = np.linspace(0, 2 * np.pi, n, endpoint=False)
    r = 10 + rng.normal(0, 0.02, n)
    pts[:, 0] = (-np.sin(ang) * r).astype(np.float32)
    pts[:, 2] = (np.cos(ang) * r).astype(np.float32)
    pts[:, 1] = -1.0
    pts[:, 3] = np.repeat(np.arange(len(sizes)), sizes) + 0.05
    s = oracle.scanreg()
    s.process(pts, sizes)
    assert s.cloud("full").shape[0] == n
    assert s.cloud("sharp").shape[0] <= 12 * len(sizes)


def test_ring_binning_restatement_equals_compiled_reference(oracle, scene):
    """MultiScanRegistration::process (unmodified reference adapter compiled against oracle/shim/ros, recorded in
    golden/multiscan_vlp16_hdl64.npz) vs the CPU restatement: binned cloud, ring sizes and the extracted features are
    bit-identical."""
    from loam_velodyne_b200 import synth
    g = _golden("multiscan_vlp16_hdl64.npz")
    for key, lidar, bounds, jitter in (("vlp16", synth.Lidar.vlp16(), (-15.0, 15.0, 16), 0.0),
                                       ("hdl64", synth.Lidar.hdl64(), (-24.9, 2.0, 64), 0.15)):
        pts, rs = synth.make_sweep(scene, lidar, 2, yaw_rate=math.radians(5.0))
        raw = synth.raw_cloud_from_sweep(pts, rs, n_bad=37, seed=5, elev_jitter_deg=jitter)
        assert_input(raw, g, f"{key}/raw")
        a = oracle.multiscan(*bounds)
        pa, sa = a.process(raw)
        np.testing.assert_array_equal(sa, g[f"{key}/sizes"])
        assert_golden(pa, g, f"{key}/binned")
        assert pa.shape[0] > 0.9 * pts.shape[0]
        for name in ("sharp", "less_sharp", "flat", "less_flat"):
            assert_golden(a.cloud(name), g, f"{key}/{name}")
        if jitter == 0.0:
            # exact ring geometry: every point returns to the ring it was cast from, in firing order
            np.testing.assert_array_equal(sa, rs)
            np.testing.assert_array_equal(np.floor(pa[:, 3]).astype(np.int32), np.repeat(np.arange(len(rs)), rs))


def test_ring_binning_restatement_matches_golden(oracle):
    """Committed output of the reference's own MultiScanRegistration::process (tests/golden/make_golden.py)."""
    g = np.load(os.path.join(HERE, "golden", "multiscan_vlp16_600.npz"))
    ms = oracle.multiscan(-15.0, 15.0, 16)
    binned, sizes = ms.process(g["raw"])
    np.testing.assert_array_equal(sizes, g["sizes"])
    np.testing.assert_array_equal(binned, g["binned"])
    np.testing.assert_array_equal(ms.cloud("sharp"), g["sharp"])
    np.testing.assert_array_equal(ms.cloud("flat"), g["flat"])


def test_transform_maintenance(oracle):
    """BasicTransformMaintenance: restatement == compiled reference (golden/transform_maintenance.npz) == the library's
    drop-in class, bit for bit (host-only arithmetic; the drop-in shares its association routine with
    BasicLaserMapping's pose prediction)."""
    from loam_velodyne_b200 import api
    g = _golden("transform_maintenance.npz")
    rng = np.random.RandomState(21)
    inputs = []
    for k in range(200):
        sum6 = np.concatenate([rng.uniform(-0.6, 0.6, 3), rng.uniform(-40, 40, 3)]).astype(np.float32)
        bef6 = (sum6 + np.concatenate([rng.normal(0, 0.02, 3), rng.normal(0, 0.5, 3)])).astype(np.float32)
        aft6 = (bef6 + np.concatenate([rng.normal(0, 0.01, 3), rng.normal(0, 0.2, 3)])).astype(np.float32)
        inputs.append(np.stack([sum6, bef6, aft6]))
        r = g["mapped"][k]
        np.testing.assert_array_equal(oracle.transform_maintenance(sum6, bef6, aft6), r)
        np.testing.assert_array_equal(api.transform_maintenance(sum6, bef6, aft6), r)
        assert np.isfinite(r).all()
    assert_input(np.stack(inputs), g, "inputs")
    # identity correction: mapped == odometry pose
    p = np.array([0.1, -0.2, 0.05, 1.0, 2.0, 3.0], np.float32)
    np.testing.assert_allclose(g["identity_out"], p, rtol=0, atol=2e-6)
    np.testing.assert_array_equal(oracle.transform_maintenance(p, p, p), g["identity_out"])
