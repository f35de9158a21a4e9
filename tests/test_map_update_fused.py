"""The end-of-sweep map update in its single-cluster form (csrc/mapstore.cuh: store_front_cluster_kernel, the run count
of store_voxel_merge_kernel, the index cleared by store_live_count_kernel and built by store_index_kernel) against the
multi-launch chain it replaces, which LOAM_B200_SPLIT_MAP_UPDATE=1 at context creation selects for every sweep: the
same poses and the same map points, bit for bit.

Which sweeps take which form: S = the stack points inserted + the raw (seeded, never filtered) map points of the cubes in
view.  The first sweep against a freshly seeded 1 M-point map has S far above the single-cluster limit (65 536) and takes
the multi-launch chain in both runs; later sweeps of that map, and every sweep of the VLP-16 streams, fit one cluster.
On the fast grid-roll trajectory cubes with raw seed points keep entering the view, so S there includes raw points
(store_front_cluster_kernel<false>)."""
import math
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SPLIT_ENV = "LOAM_B200_SPLIT_MAP_UPDATE"


def _run(split, corner, surf, sweeps, stream):
    from loam_velodyne_b200 import api
    if split:
        os.environ[SPLIT_ENV] = "1"
    try:
        p = api.Pipeline()
        p.seed_map(corner, surf)
        if stream:
            poses = [(ok, od, aft) for ok, od, aft in p.run_stream(sweeps)]
        else:
            poses = [p.sweep(pts, rs)[:3] for pts, rs in sweeps]
        p.sync()
        maps = {k: p.mapping.cloud(k) for k in ("corner_cubes", "surf_cubes")}
        del p
    finally:
        os.environ.pop(SPLIT_ENV, None)
    return poses, maps


def _case(name):
    from loam_velodyne_b200 import synth
    if name == "vlp16_200k_stream":
        sc = synth.make_scene()
        lidar = synth.Lidar.vlp16()
        corner, surf = synth.make_map(sc, 200_000)
        return corner, surf, [synth.make_sweep(sc, lidar, i, yaw_rate=math.radians(5.0)) for i in range(8)], True
    if name == "hdl64_1m":
        sc = synth.make_scene()
        lidar = synth.Lidar.hdl64()
        corner, surf = synth.make_map(sc, 1_000_000)
        return corner, surf, [synth.make_sweep(sc, lidar, i, yaw_rate=math.radians(5.0)) for i in range(10)], False
    if name == "grid_roll_raw_cubes":  # test_map_grid_roll_and_drop's trajectory: 30 m/s along x, the grid rolls twice
        sc = synth.make_scene(seed=3, extent=160.0)
        lidar = synth.Lidar(16, 600, -15.0, 15.0)
        corner, surf = synth.make_map(sc, 150_000, window=150.0)
        return corner, surf, [synth.make_sweep(sc, lidar, i, v=(30.0, 0.0, 0.0), yaw_rate=0.0) for i in range(45)], False
    raise ValueError(name)


@pytest.mark.parametrize("name", ["vlp16_200k_stream", "hdl64_1m", "grid_roll_raw_cubes"])
def test_single_cluster_update_equals_multi_launch_chain(build_libs, name):
    corner, surf, sweeps, stream = _case(name)
    poses_a, maps_a = _run(False, corner, surf, sweeps, stream)
    poses_b, maps_b = _run(True, corner, surf, sweeps, stream)
    assert len(poses_a) == len(poses_b) == len(sweeps)
    for i, ((ok_a, od_a, aft_a), (ok_b, od_b, aft_b)) in enumerate(zip(poses_a, poses_b)):
        assert ok_a == ok_b, i
        assert np.array_equal(od_a, od_b), (i, od_a, od_b)
        assert np.array_equal(aft_a, aft_b), (i, aft_a, aft_b)
    for k in ("corner_cubes", "surf_cubes"):
        assert maps_a[k].shape[0] > 0, k
        assert np.array_equal(maps_a[k], maps_b[k]), k
