"""Regenerates tests/golden/* from oracle/_ref (the UNMODIFIED reference sources compiled against oracle/shim).

Run where `make -C oracle ref` has built oracle/_ref from the reference sources:   python tests/golden/make_golden.py
The fixtures are small on purpose so they can live in git; they pin
 * the feature clouds of BasicScanRegistration::processScanlines,
 * the odometry / mapping poses of registration -> odometry -> mapping runs (several sensor geometries, ragged rings,
   non-default RegistrationParams, tight iteration budgets),
 * k-NN, VoxelGrid and the dense solves on fixed inputs,
 * the ring-binning front end (MultiScanRegistration::process) on jittered, defect-laden raw clouds,
 * BasicTransformMaintenance on random poses,
 * the loam:: symbols the reference's ROS adapters need from the library that replaces the Basic* classes.
pipeline_vlp16_600.npz, pieces.npz and multiscan_vlp16_600.npz hold their inputs and outputs whole.  The other fixtures
do not store inputs that loam_velodyne_b200.synth regenerates deterministically, only their SHA-256, so a test can tell
a changed generator from a changed result; their arrays of more than FULL_MAX_ROWS rows are stored as SHA-256 + shape
+ SAMPLE_ROWS evenly spaced rows (bit-exact comparison, readable diff on the sampled rows).
"""
import glob
import hashlib
import math
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from loam_velodyne_b200 import synth  # noqa: E402
from oracle import pydriver  # noqa: E402
from test_oracle import VARIANTS  # noqa: E402  (the cases the restatement is checked on)

HERE = os.path.dirname(os.path.abspath(__file__))
FULL_MAX_ROWS = 32
SAMPLE_ROWS = 16

FEATURES = ("sharp", "less_sharp", "flat", "less_flat")
ADAPTERS = ["ScanRegistration", "MultiScanRegistration", "LaserOdometry", "LaserMapping", "TransformMaintenance"]


def sample_rows(n):
    return np.unique(np.linspace(0, n - 1, SAMPLE_ROWS).astype(np.int64))


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def put(out, key, a):
    """Store `a` under `key` whole, or as key__sha256 / key__shape / key__sample when it is large."""
    a = np.ascontiguousarray(a)
    if a.ndim == 0 or a.shape[0] <= FULL_MAX_ROWS:
        out[key] = a
    else:
        out[key + "__sha256"] = np.array(sha256(a))
        out[key + "__shape"] = np.array(a.shape, np.int64)
        out[key + "__sample"] = a[sample_rows(a.shape[0])]


def pipeline_vlp16_600(ref, scene):
    lidar = synth.Lidar(16, 600, -15.0, 15.0)
    corner, surf = synth.make_map(scene, 40_000)
    pipe = ref.pipeline()
    pipe.seed_map(corner, surf)
    out = {"map_corner": corner, "map_surf": surf}
    for i in range(6):
        pts, rs = synth.make_sweep(scene, lidar, i, yaw_rate=math.radians(5.0))
        ok, odom, aft, _ = pipe.sweep(pts, rs)
        out[f"pts{i}"] = pts
        out[f"rings{i}"] = rs
        out[f"odom{i}"] = odom
        out[f"aft{i}"] = aft
        if i in (0, 3):
            for name in FEATURES:
                out[f"{name}{i}"] = pipe.scanreg.cloud(name)
    out["final_corner_cubes"] = pipe.mapping.cloud("corner_cubes")
    out["final_surf_cubes_n"] = np.array([pipe.mapping.cloud("surf_cubes").shape[0]])
    np.savez_compressed(os.path.join(HERE, "pipeline_vlp16_600.npz"), **out)
    return corner, surf, out["pts2"]


def pipeline_vlp16_900_live(ref, scene):
    lidar = synth.Lidar(16, 900, -15.0, 15.0)
    corner, surf = synth.make_map(scene, 60_000)
    pipe = ref.pipeline()
    pipe.seed_map(corner, surf)
    out = {"map_corner__sha256": np.array(sha256(corner)), "map_surf__sha256": np.array(sha256(surf))}
    for i in range(5):
        pts, rs = synth.make_sweep(scene, lidar, 20 + i, yaw_rate=math.radians(-7.0), v=(0.3, 0.0, 1.5))
        ok, odom, aft, _ = pipe.sweep(pts, rs)
        out[f"pts{i}__sha256"] = np.array(sha256(pts))
        out[f"ok{i}"] = np.array(ok)
        out[f"odom{i}"] = odom
        out[f"aft{i}"] = aft
        for name in FEATURES:
            put(out, f"{name}{i}", pipe.scanreg.cloud(name))
        for name in ("last_corner", "last_surf"):
            put(out, f"{name}{i}", pipe.odom.cloud(name))
    np.savez_compressed(os.path.join(HERE, "pipeline_vlp16_900_live.npz"), **out)


def pipeline_variants(ref, scene):
    out = {}
    corner, surf = synth.make_map(scene, 40_000)
    out["map_corner__sha256"] = np.array(sha256(corner))
    out["map_surf__sha256"] = np.array(sha256(surf))
    for variant, (R, A, lo, hi, yaw, v, max_range, reg, (oi, mi)) in sorted(VARIANTS.items()):
        lidar = synth.Lidar(R, A, lo, hi)
        pipe = ref.pipeline(odom_iter=oi, map_iter=mi)
        if reg:
            pipe.scanreg.configure(**reg)
        pipe.seed_map(corner, surf)
        for i in range(4):
            pts, rs = synth.make_sweep(scene, lidar, 5 + i, yaw_rate=math.radians(yaw), v=v, max_range=max_range)
            ok, odom, aft, _ = pipe.sweep(pts, rs)
            out[f"{variant}/pts{i}__sha256"] = np.array(sha256(pts))
            out[f"{variant}/ok{i}"] = np.array(ok)
            out[f"{variant}/odom{i}"] = odom
            out[f"{variant}/aft{i}"] = aft
            for name in FEATURES:
                put(out, f"{variant}/{name}{i}", pipe.scanreg.cloud(name))
        for name in ("corner_cubes", "surf_cubes"):
            put(out, f"{variant}/{name}", pipe.mapping.cloud(name))
    np.savez_compressed(os.path.join(HERE, "pipeline_variants.npz"), **out)


def pieces(ref, corner, surf, pts2):
    rng = np.random.RandomState(11)
    q = surf[rng.randint(0, surf.shape[0], 400)].copy()
    q[:, :3] += rng.normal(0, 0.3, (400, 3)).astype(np.float32)
    idx5, d5 = ref.knn(surf, q, 5)
    idx1, d1 = ref.knn(corner, q, 1)
    vox = ref.voxel_grid(pts2, 0.4)
    A = rng.normal(size=(6, 6)).astype(np.float32)
    A = (A @ A.T + 6 * np.eye(6)).astype(np.float32)
    b = rng.normal(size=6).astype(np.float32)
    x = ref.qr_solve6(A, b)
    ev, V = ref.eig_sym(A)
    A3 = A[:3, :3].copy()
    ev3, V3 = ref.eig_sym(A3)
    P5 = (surf[1000:1005, :3] + rng.normal(0, 0.01, (5, 3))).astype(np.float32)
    x53 = ref.lsq53(P5)
    np.savez_compressed(os.path.join(HERE, "pieces.npz"), knn_pts=surf, knn_corner=corner, knn_q=q, knn_idx5=idx5,
                        knn_d5=d5, knn_idx1=idx1, knn_d1=d1, vox_in=pts2, vox_out=vox, A=A, b=b, x=x, ev=ev,
                        V=V, ev3=ev3, V3=V3, P5=P5, x53=x53)


def multiscan(ref, scene):
    # ring-binning front end: MultiScanRegistration::process (the reference's ROS adapter compiled against oracle/shim/ros)
    lid = synth.Lidar(16, 600, -15.0, 15.0)
    pts_f, rs_f = synth.make_sweep(scene, lid, 2, yaw_rate=math.radians(5.0))
    raw = synth.raw_cloud_from_sweep(pts_f, rs_f, n_bad=25, seed=9, elev_jitter_deg=0.2)
    ms = ref.multiscan(-15.0, 15.0, 16)
    binned, sizes = ms.process(raw)
    np.savez_compressed(os.path.join(HERE, "multiscan_vlp16_600.npz"), raw=raw, binned=binned, sizes=sizes,
                        sharp=ms.cloud("sharp"), flat=ms.cloud("flat"))
    # VLP-16 on its exact ring geometry and HDL-64 with jittered elevations, raw clouds regenerated by the tests
    out = {}
    for name, lidar, bounds, jitter in (("vlp16", synth.Lidar.vlp16(), (-15.0, 15.0, 16), 0.0),
                                        ("hdl64", synth.Lidar.hdl64(), (-24.9, 2.0, 64), 0.15)):
        pts, rs = synth.make_sweep(scene, lidar, 2, yaw_rate=math.radians(5.0))
        raw = synth.raw_cloud_from_sweep(pts, rs, n_bad=37, seed=5, elev_jitter_deg=jitter)
        ms = ref.multiscan(*bounds)
        binned, sizes = ms.process(raw)
        out[f"{name}/raw__sha256"] = np.array(sha256(raw))
        out[f"{name}/sizes"] = sizes
        put(out, f"{name}/binned", binned)
        for f in FEATURES:
            put(out, f"{name}/{f}", ms.cloud(f))
    np.savez_compressed(os.path.join(HERE, "multiscan_vlp16_hdl64.npz"), **out)


def transform_maintenance(ref):
    rng = np.random.RandomState(21)
    ins, outs = [], []
    for _ in range(200):
        sum6 = np.concatenate([rng.uniform(-0.6, 0.6, 3), rng.uniform(-40, 40, 3)]).astype(np.float32)
        bef6 = (sum6 + np.concatenate([rng.normal(0, 0.02, 3), rng.normal(0, 0.5, 3)])).astype(np.float32)
        aft6 = (bef6 + np.concatenate([rng.normal(0, 0.01, 3), rng.normal(0, 0.2, 3)])).astype(np.float32)
        ins.append(np.stack([sum6, bef6, aft6]))
        outs.append(ref.transform_maintenance(sum6, bef6, aft6))
    p = np.array([0.1, -0.2, 0.05, 1.0, 2.0, 3.0], np.float32)
    np.savez_compressed(os.path.join(HERE, "transform_maintenance.npz"), inputs__sha256=np.array(sha256(np.stack(ins))),
                        mapped=np.stack(outs), identity_out=ref.transform_maintenance(p, p, p))


def dropin_symbols(ref_src):
    """The loam:: symbols the reference's five ROS adapters leave undefined when compiled UNCHANGED against the product's
    replacement headers (the overlay tests/test_dropin.py builds) -- what libloam_b200.so has to export."""
    host = os.path.join(ROOT, "loam_velodyne_b200", "csrc", "host")
    with tempfile.TemporaryDirectory() as d:
        inc = os.path.join(d, "loam_velodyne")
        os.mkdir(inc)
        for f in glob.glob(os.path.join(ref_src, "include", "loam_velodyne", "*")):
            shutil.copyfile(f, os.path.join(inc, os.path.basename(f)))
        for f in glob.glob(os.path.join(host, "loam_velodyne", "*.h")):
            shutil.copyfile(f, os.path.join(inc, os.path.basename(f)))
        flags = ["-std=c++14", "-fPIC", f"-I{d}", f"-I{host}", f"-I{host}/compat", f"-I{ROOT}/include",
                 f"-I{ROOT}/oracle/shim", f"-I{ref_src}/src/lib"]
        needed, defined = set(), set()
        for name in ADAPTERS:
            obj = os.path.join(d, name + ".o")
            subprocess.run(["g++", "-c", *flags, "-o", obj, os.path.join(ref_src, "src", "lib", name + ".cpp")], check=True)
            nm = lambda *opt: subprocess.run(["nm", *opt, "--format=just-symbols", obj], check=True, capture_output=True,
                                             text=True).stdout.split()
            needed |= {s for s in nm("-u") if s.startswith(("_ZN4loam", "_ZNK4loam"))}
            defined |= set(nm("--defined-only"))
    with open(os.path.join(HERE, "dropin_symbols.txt"), "w") as fh:
        fh.write("".join(s + "\n" for s in sorted(needed - defined)))


def main():
    ref = pydriver.load("reference")
    assert ref.kind == "reference"
    scene = synth.make_scene()
    corner, surf, pts2 = pipeline_vlp16_600(ref, scene)
    pieces(ref, corner, surf, pts2)
    multiscan(ref, scene)
    pipeline_vlp16_900_live(ref, scene)
    pipeline_variants(ref, scene)
    transform_maintenance(ref)
    dropin_symbols(pydriver.reference_source())
    print("golden fixtures written:", sorted(os.listdir(HERE)))


if __name__ == "__main__":
    main()
