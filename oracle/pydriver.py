"""TEST INFRASTRUCTURE -- ctypes binding of oracle/driver_api.h (not part of the shipped product).

``load("reference")`` -> oracle/_ref/libloam_ref.so  (the unmodified reference sources compiled against oracle/shim)
``load("restatement")`` -> oracle/liboracle.so       (the CPU restatement, oracle/loam_oracle.cpp)
``fast=True`` picks the -O3 builds used for the timed CPU baseline.
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

_F = C.POINTER(C.c_float)
_I = C.POINTER(C.c_int)
_D = C.POINTER(C.c_double)


def _fp(a):
    return a.ctypes.data_as(_F)


def _ip(a):
    return a.ctypes.data_as(_I)


def _pts(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] != 4:
        a = a.reshape(-1, 4)
    return a


def lib_path(kind: str, fast: bool = False) -> str:
    if kind == "reference":
        return os.path.join(HERE, "_ref", "libloam_ref_fast.so" if fast else "libloam_ref.so")
    return os.path.join(HERE, "liboracle_fast.so" if fast else "liboracle.so")


def available(kind: str, fast: bool = False) -> bool:
    return os.path.exists(lib_path(kind, fast))


def reference_source():
    """The reference source tree oracle/_ref was compiled from (`make ref` records it), or None where it is absent."""
    p = os.path.join(HERE, "_ref", "source_dir")
    if not os.path.exists(p):
        return None
    with open(p) as fh:
        d = fh.read().strip()
    return d if os.path.isdir(os.path.join(d, "src", "lib")) else None


_cache = {}


def load(kind: str = "reference", fast: bool = False) -> "Driver":
    key = (kind, fast)
    if key not in _cache:
        _cache[key] = Driver(lib_path(kind, fast))
    return _cache[key]


def best(fast: bool = False) -> "Driver":
    """The strongest checker present: the compiled reference if it travelled here, else the restatement."""
    return load("reference" if available("reference", fast) else "restatement", fast)


class Driver:
    def __init__(self, path: str):
        self.path = path
        L = self.L = C.CDLL(path)
        vp = C.c_void_p
        sig = {
            "loamdrv_kind": (C.c_char_p, []),
            "loamdrv_scanreg_create": (vp, []),
            "loamdrv_scanreg_destroy": (None, [vp]),
            "loamdrv_scanreg_configure": (None, [vp, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float]),
            "loamdrv_scanreg_process": (C.c_int, [vp, _F, _I, C.c_int]),
            "loamdrv_scanreg_cloud_size": (C.c_int, [vp, C.c_int]),
            "loamdrv_scanreg_cloud_copy": (None, [vp, C.c_int, _F]),
            "loamdrv_transform_maintenance": (None, [_F, _F, _F, _F]),
            "loamdrv_multiscan_create": (vp, [C.c_float, C.c_float, C.c_int]),
            "loamdrv_multiscan_destroy": (None, [vp]),
            "loamdrv_multiscan_process": (C.c_int, [vp, _F, C.c_int]),
            "loamdrv_multiscan_binned": (None, [vp, _F, _I]),
            "loamdrv_multiscan_cloud_size": (C.c_int, [vp, C.c_int]),
            "loamdrv_multiscan_cloud_copy": (None, [vp, C.c_int, _F]),
            "loamdrv_odom_create": (vp, [C.c_float, C.c_int]),
            "loamdrv_odom_destroy": (None, [vp]),
            "loamdrv_odom_set_inputs": (None, [vp, _F, C.c_int, _F, C.c_int, _F, C.c_int, _F, C.c_int, _F, C.c_int]),
            "loamdrv_odom_process": (None, [vp]),
            "loamdrv_odom_full_to_end": (None, [vp]),
            "loamdrv_odom_get_twist": (None, [vp, C.c_int, _F]),
            "loamdrv_odom_cloud_size": (C.c_int, [vp, C.c_int]),
            "loamdrv_odom_cloud_copy": (None, [vp, C.c_int, _F]),
            "loamdrv_map_create": (vp, [C.c_float, C.c_int]),
            "loamdrv_map_destroy": (None, [vp]),
            "loamdrv_map_seed": (None, [vp, C.c_int, _F, C.c_int]),
            "loamdrv_map_set_inputs": (None, [vp, _F, C.c_int, _F, C.c_int, _F, C.c_int]),
            "loamdrv_map_update_odometry": (None, [vp, _F]),
            "loamdrv_map_process": (C.c_int, [vp]),
            "loamdrv_map_get_twist": (None, [vp, C.c_int, _F]),
            "loamdrv_map_cloud_size": (C.c_int, [vp, C.c_int]),
            "loamdrv_map_cloud_copy": (None, [vp, C.c_int, _F]),
            "loamdrv_pipeline_create": (vp, [C.c_float, C.c_int, C.c_int]),
            "loamdrv_pipeline_destroy": (None, [vp]),
            "loamdrv_pipeline_seed_map": (None, [vp, C.c_int, _F, C.c_int]),
            "loamdrv_pipeline_sweep": (C.c_int, [vp, _F, _I, C.c_int, _F, _F, _D]),
            "loamdrv_pipeline_scanreg": (vp, [vp]),
            "loamdrv_pipeline_odom": (vp, [vp]),
            "loamdrv_pipeline_map": (vp, [vp]),
            "loamdrv_knn": (C.c_int, [_F, C.c_int, _F, C.c_int, C.c_int, _I, _F]),
            "loamdrv_kdtree_build_seconds": (C.c_double, [_F, C.c_int]),
            "loamdrv_voxel_grid": (C.c_int, [_F, C.c_int, C.c_float, _F]),
            "loamdrv_qr_solve6": (None, [_F, _F, _F]),
            "loamdrv_eig_sym": (None, [_F, C.c_int, _F, _F]),
            "loamdrv_lsq53": (None, [_F, _F]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        self.kind = L.loamdrv_kind().decode()
        if self.kind == "restatement":
            # per-iteration hooks only the restatement offers (the reference classes cannot be paused mid-process)
            _S = C.POINTER(C.c_int8)
            L.loamorc_odom_iteration.restype = C.c_int
            L.loamorc_odom_iteration.argtypes = [vp, C.c_int, _F, _F, _S, _F, _F]
            L.loamorc_odom_indices.restype = None
            L.loamorc_odom_indices.argtypes = [vp, _I]
            L.loamorc_odom_set_last.restype = None
            L.loamorc_odom_set_last.argtypes = [vp, _F, C.c_int, _F, C.c_int]
            L.loamorc_map_set.restype = None
            L.loamorc_map_set.argtypes = [vp, _F, C.c_int, _F, C.c_int, _F, C.c_int, _F, C.c_int]
            L.loamorc_map_iteration.restype = C.c_int
            L.loamorc_map_iteration.argtypes = [vp, _F, _F, _S, _F, _F]

    # ---- generic cloud getter
    def _cloud(self, size_fn, copy_fn, h, which):
        n = size_fn(h, which)
        out = np.empty((n, 4), dtype=np.float32)
        if n:
            copy_fn(h, which, _fp(out))
        return out

    # ---- pieces
    def knn(self, pts, queries, k):
        pts = _pts(pts)
        queries = _pts(queries)
        idx = np.empty((queries.shape[0], k), dtype=np.int32)
        d2 = np.empty((queries.shape[0], k), dtype=np.float32)
        self.L.loamdrv_knn(_fp(pts), pts.shape[0], _fp(queries), queries.shape[0], k, _ip(idx), _fp(d2))
        return idx, d2

    def kdtree_build_seconds(self, pts):
        pts = _pts(pts)
        return self.L.loamdrv_kdtree_build_seconds(_fp(pts), pts.shape[0])

    def voxel_grid(self, pts, leaf):
        pts = _pts(pts)
        out = np.empty_like(pts)
        n = self.L.loamdrv_voxel_grid(_fp(pts), pts.shape[0], leaf, _fp(out))
        return out[:n].copy()

    def qr_solve6(self, A, b):
        A = np.ascontiguousarray(A, dtype=np.float32)
        b = np.ascontiguousarray(b, dtype=np.float32)
        x = np.empty(6, dtype=np.float32)
        self.L.loamdrv_qr_solve6(_fp(A), _fp(b), _fp(x))
        return x

    def eig_sym(self, A):
        A = np.ascontiguousarray(A, dtype=np.float32)
        n = A.shape[0]
        ev = np.empty(n, dtype=np.float32)
        V = np.empty((n, n), dtype=np.float32)
        self.L.loamdrv_eig_sym(_fp(A), n, _fp(ev), _fp(V))
        return ev, V.T.copy()  # V stored column-major -> columns are eigenvectors

    def lsq53(self, A):
        A = np.ascontiguousarray(A, dtype=np.float32)
        x = np.empty(3, dtype=np.float32)
        self.L.loamdrv_lsq53(_fp(A), _fp(x))
        return x

    # ---- objects
    def transform_maintenance(self, sum6, bef6, aft6):
        a = [np.ascontiguousarray(v, dtype=np.float32).reshape(6) for v in (sum6, bef6, aft6)]
        out = np.zeros(6, np.float32)
        self.L.loamdrv_transform_maintenance(_fp(a[0]), _fp(a[1]), _fp(a[2]), _fp(out))
        return out

    def multiscan(self, lower_deg, upper_deg, n_rings):
        return MultiScan(self, lower_deg, upper_deg, n_rings)

    def scanreg(self):
        return ScanReg(self)

    def odom(self, scan_period=0.1, max_iter=25):
        return Odom(self, scan_period, max_iter)

    def mapping(self, scan_period=0.1, max_iter=10):
        return Mapping(self, scan_period, max_iter)

    def pipeline(self, scan_period=0.1, odom_iter=25, map_iter=10):
        return Pipeline(self, scan_period, odom_iter, map_iter)


class ScanReg:
    NAMES = {"full": 0, "sharp": 1, "less_sharp": 2, "flat": 3, "less_flat": 4}

    def __init__(self, drv, handle=None):
        self.d = drv
        self.own = handle is None
        self.h = handle if handle is not None else drv.L.loamdrv_scanreg_create()

    def __del__(self):
        if getattr(self, "own", False) and self.h:
            self.d.L.loamdrv_scanreg_destroy(self.h)
            self.h = None

    def configure(self, scan_period=0.1, n_regions=6, curv_region=5, max_sharp=2, max_flat=4, less_flat_leaf=0.2,
                  curv_thr=0.1):
        self.d.L.loamdrv_scanreg_configure(self.h, scan_period, n_regions, curv_region, max_sharp, max_flat,
                                           less_flat_leaf, curv_thr)

    def process(self, pts, ring_sizes):
        pts = _pts(pts)
        ring_sizes = np.ascontiguousarray(ring_sizes, dtype=np.int32)
        return self.d.L.loamdrv_scanreg_process(self.h, _fp(pts), _ip(ring_sizes), ring_sizes.shape[0])

    def cloud(self, name):
        return self.d._cloud(self.d.L.loamdrv_scanreg_cloud_size, self.d.L.loamdrv_scanreg_cloud_copy, self.h,
                             self.NAMES[name])


class MultiScan:
    """Ring-binning front end (MultiScanRegistration::process, MultiScanRegistration.cpp:160-238) + registration."""
    NAMES = ScanReg.NAMES

    def __init__(self, drv, lower_deg, upper_deg, n_rings):
        self.d = drv
        self.n_rings = n_rings
        self.h = drv.L.loamdrv_multiscan_create(lower_deg, upper_deg, n_rings)

    def __del__(self):
        if getattr(self, "h", None):
            self.d.L.loamdrv_multiscan_destroy(self.h)
            self.h = None

    def process(self, xyz):
        """xyz: n x 3 sensor-frame points in arrival order -> (ring-ordered n_kept x 4 cloud, ring sizes)."""
        a = np.ascontiguousarray(xyz, dtype=np.float32)
        kept = self.d.L.loamdrv_multiscan_process(self.h, _fp(a), a.shape[0])
        out = np.empty((kept, 4), np.float32)
        sizes = np.zeros(self.n_rings, np.int32)
        self.d.L.loamdrv_multiscan_binned(self.h, _fp(out), _ip(sizes))
        return out, sizes

    def cloud(self, name):
        return self.d._cloud(self.d.L.loamdrv_multiscan_cloud_size, self.d.L.loamdrv_multiscan_cloud_copy, self.h,
                             self.NAMES[name])


class Odom:
    NAMES = {"last_corner": 0, "last_surf": 1, "full": 2}

    def __init__(self, drv, scan_period=0.1, max_iter=25, handle=None):
        self.d = drv
        self.own = handle is None
        self.h = handle if handle is not None else drv.L.loamdrv_odom_create(scan_period, max_iter)

    def __del__(self):
        if getattr(self, "own", False) and self.h:
            self.d.L.loamdrv_odom_destroy(self.h)
            self.h = None

    def set_inputs(self, sharp, less_sharp, flat, less_flat, full):
        a = [_pts(x) for x in (sharp, less_sharp, flat, less_flat, full)]
        self.d.L.loamdrv_odom_set_inputs(self.h, _fp(a[0]), a[0].shape[0], _fp(a[1]), a[1].shape[0], _fp(a[2]),
                                         a[2].shape[0], _fp(a[3]), a[3].shape[0], _fp(a[4]), a[4].shape[0])

    def process(self):
        self.d.L.loamdrv_odom_process(self.h)

    def full_to_end(self):
        self.d.L.loamdrv_odom_full_to_end(self.h)

    def twist(self, which):
        out = np.empty(6, dtype=np.float32)
        self.d.L.loamdrv_odom_get_twist(self.h, {"transform": 0, "sum": 1}[which], _fp(out))
        return out

    def cloud(self, name):
        return self.d._cloud(self.d.L.loamdrv_odom_cloud_size, self.d.L.loamdrv_odom_cloud_copy, self.h,
                             self.NAMES[name])


class Mapping:
    NAMES = {"full": 0, "surround_ds": 1, "corner_from_map": 2, "surf_from_map": 3, "corner_stack_ds": 4,
             "surf_stack_ds": 5, "corner_cubes": 6, "surf_cubes": 7}

    def __init__(self, drv, scan_period=0.1, max_iter=10, handle=None):
        self.d = drv
        self.own = handle is None
        self.h = handle if handle is not None else drv.L.loamdrv_map_create(scan_period, max_iter)

    def __del__(self):
        if getattr(self, "own", False) and self.h:
            self.d.L.loamdrv_map_destroy(self.h)
            self.h = None

    def seed(self, corner, surf):
        c, s = _pts(corner), _pts(surf)
        self.d.L.loamdrv_map_seed(self.h, 0, _fp(c), c.shape[0])
        self.d.L.loamdrv_map_seed(self.h, 1, _fp(s), s.shape[0])

    def set_inputs(self, corner_last, surf_last, full):
        a = [_pts(x) for x in (corner_last, surf_last, full)]
        self.d.L.loamdrv_map_set_inputs(self.h, _fp(a[0]), a[0].shape[0], _fp(a[1]), a[1].shape[0], _fp(a[2]),
                                        a[2].shape[0])

    def update_odometry(self, sum6):
        s = np.ascontiguousarray(sum6, dtype=np.float32)
        self.d.L.loamdrv_map_update_odometry(self.h, _fp(s))

    def process(self):
        return bool(self.d.L.loamdrv_map_process(self.h))

    def twist(self, which):
        out = np.empty(6, dtype=np.float32)
        self.d.L.loamdrv_map_get_twist(self.h, {"aft": 0, "bef": 1, "tobe": 2}[which], _fp(out))
        return out

    def cloud(self, name):
        return self.d._cloud(self.d.L.loamdrv_map_cloud_size, self.d.L.loamdrv_map_cloud_copy, self.h,
                             self.NAMES[name])


def map_iteration(drv, corner_map, surf_map, corner_q, surf_q, tobe6):
    """One correspondence + normal-equation pass of the scan-to-map loop at pose tobe6 (restatement only)."""
    m = drv.mapping()
    a = [_pts(x) for x in (corner_map, surf_map, corner_q, surf_q)]
    drv.L.loamorc_map_set(m.h, _fp(a[0]), a[0].shape[0], _fp(a[1]), a[1].shape[0], _fp(a[2]), a[2].shape[0], _fp(a[3]),
                          a[3].shape[0])
    nq = a[2].shape[0] + a[3].shape[0]
    coeff = np.zeros((nq, 4), np.float32)
    sel = np.zeros(nq, np.int8)
    AtA = np.zeros((6, 6), np.float32)
    AtB = np.zeros(6, np.float32)
    t = np.ascontiguousarray(tobe6, dtype=np.float32)
    n = drv.L.loamorc_map_iteration(m.h, _fp(t), _fp(coeff), sel.ctypes.data_as(C.POINTER(C.c_int8)), _fp(AtA), _fp(AtB))
    return {"n_selected": n, "coeff": coeff, "selected": sel, "AtA": AtA, "AtB": AtB}


class OdomIterator:
    """Steps the scan-to-scan loop one iteration at a time (restatement only)."""

    def __init__(self, drv, last_corner, last_surf, sharp, flat, scan_period=0.1):
        self.d = drv
        self.o = drv.odom(scan_period, 25)
        lc, ls = _pts(last_corner), _pts(last_surf)
        drv.L.loamorc_odom_set_last(self.o.h, _fp(lc), lc.shape[0], _fp(ls), ls.shape[0])
        empty = np.zeros((0, 4), np.float32)
        self.o.set_inputs(sharp, empty, flat, empty, empty)
        self.nq = _pts(sharp).shape[0] + _pts(flat).shape[0]

    def iterate(self, it, transform6):
        coeff = np.zeros((self.nq, 4), np.float32)
        sel = np.zeros(self.nq, np.int8)
        AtA = np.zeros((6, 6), np.float32)
        AtB = np.zeros(6, np.float32)
        t = np.ascontiguousarray(transform6, dtype=np.float32)
        n = self.d.L.loamorc_odom_iteration(self.o.h, it, _fp(t), _fp(coeff), sel.ctypes.data_as(C.POINTER(C.c_int8)),
                                            _fp(AtA), _fp(AtB))
        ind = np.full((self.nq, 3), -1, np.int32)
        self.d.L.loamorc_odom_indices(self.o.h, _ip(ind))
        return {"n_selected": n, "coeff": coeff, "selected": sel, "AtA": AtA, "AtB": AtB, "ind": ind}


class Pipeline:
    def __init__(self, drv, scan_period=0.1, odom_iter=25, map_iter=10):
        self.d = drv
        self.h = drv.L.loamdrv_pipeline_create(scan_period, odom_iter, map_iter)
        self.scanreg = ScanReg(drv, drv.L.loamdrv_pipeline_scanreg(self.h))
        self.odom = Odom(drv, handle=drv.L.loamdrv_pipeline_odom(self.h))
        self.mapping = Mapping(drv, handle=drv.L.loamdrv_pipeline_map(self.h))

    def __del__(self):
        if getattr(self, "h", None):
            self.d.L.loamdrv_pipeline_destroy(self.h)
            self.h = None

    def seed_map(self, corner, surf):
        c, s = _pts(corner), _pts(surf)
        self.d.L.loamdrv_pipeline_seed_map(self.h, 0, _fp(c), c.shape[0])
        self.d.L.loamdrv_pipeline_seed_map(self.h, 1, _fp(s), s.shape[0])

    def sweep(self, pts, ring_sizes):
        pts = _pts(pts)
        ring_sizes = np.ascontiguousarray(ring_sizes, dtype=np.int32)
        odom = np.empty(6, dtype=np.float32)
        aft = np.empty(6, dtype=np.float32)
        st = np.zeros(5, dtype=np.float64)
        ok = self.d.L.loamdrv_pipeline_sweep(self.h, _fp(pts), _ip(ring_sizes), ring_sizes.shape[0], _fp(odom),
                                             _fp(aft), st.ctypes.data_as(_D))
        return bool(ok), odom, aft, st
