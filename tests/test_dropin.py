"""The drop-in boundary, checked the way a maintainer would use it (SURVEY.md section 8b): the reference's five ROS adapters
(src/lib/{ScanRegistration,MultiScanRegistration,LaserOdometry,LaserMapping,TransformMaintenance}.cpp) are compiled
UNCHANGED against the product's replacement headers and linked against libloam_b200.so.

The adapters include their siblings with quote includes (LaserOdometry.h: #include "BasicLaserOdometry.h"), which resolve
in the including file's directory first, so the product headers must REPLACE the reference's files (INTEGRATION.md): the
test builds exactly that overlay in a temporary directory -- the reference's include/loam_velodyne/ with the product's
loam_velodyne/*.h copied over it.  ROS itself is absent here; oracle/shim/{ros,tf,nav_msgs,sensor_msgs,
geometry_msgs,pcl_conversions} stands in for the few names the adapters mention (test infrastructure).
Compiling the adapters needs the upstream loam_velodyne source tree oracle/_ref was built from (build() records where it
lies); without it that test skips.  The link check runs everywhere: the loam:: symbols the adapters need were recorded from that build in
golden/dropin_symbols.txt (tests/golden/make_golden.py)."""
import ctypes
import glob
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "loam_velodyne_b200", "csrc", "host")
ADAPTERS = ["ScanRegistration", "MultiScanRegistration", "LaserOdometry", "LaserMapping", "TransformMaintenance"]

@pytest.fixture(scope="module")
def upstream(build_libs):
    from oracle import pydriver
    src = pydriver.reference_source()
    if src is None:
        pytest.skip("needs the upstream loam_velodyne sources oracle/_ref is built from")
    return src


@pytest.fixture(scope="module")
def overlay(tmp_path_factory, upstream):
    d = tmp_path_factory.mktemp("dropin")
    inc = d / "loam_velodyne"
    inc.mkdir()
    for f in glob.glob(os.path.join(upstream, "include", "loam_velodyne", "*")):
        shutil.copyfile(f, os.path.join(inc, os.path.basename(f)))
    replaced = []
    # the product's headers replace their upstream namesakes (copyfile: the upstream copies may be read-only)
    for f in glob.glob(os.path.join(HOST, "loam_velodyne", "*.h")):
        shutil.copyfile(f, os.path.join(inc, os.path.basename(f)))
        replaced.append(os.path.basename(f))
    assert {"BasicScanRegistration.h", "BasicLaserOdometry.h", "BasicLaserMapping.h", "BasicTransformMaintenance.h"} <= set(replaced)
    return d


def _flags(overlay, upstream):
    return ["-std=c++14", "-fPIC", f"-I{overlay}", f"-I{HOST}", f"-I{HOST}/compat", f"-I{ROOT}/include",
            f"-I{ROOT}/oracle/shim", f"-I{upstream}/src/lib"]


@pytest.mark.parametrize("name", ADAPTERS)
def test_reference_adapter_compiles_against_product_headers(overlay, upstream, name):
    r = subprocess.run(["g++", "-fsyntax-only", *_flags(overlay, upstream), os.path.join(upstream, "src", "lib", name + ".cpp")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]


def test_reference_adapters_link_against_the_product_library(build_libs):
    """Every loam:: symbol the adapters use (recorded from their build against the product headers) is exported by
    libloam_b200.so (no undefined reference)."""
    from loam_velodyne_b200 import api
    with open(os.path.join(ROOT, "tests", "golden", "dropin_symbols.txt")) as fh:
        needed = fh.read().split()
    assert len(needed) > 30
    L = ctypes.CDLL(api.LIB_PATH)
    missing = [s for s in needed if not hasattr(L, s)]
    assert not missing, f"not exported by {api.LIB_PATH}: {missing}"


def test_product_headers_do_not_redeclare_adapter_classes():
    """loam::MultiScanMapper belongs to upstream's MultiScanRegistration.h:49; a second definition in the product headers
    broke upstream's MultiScanRegistration.cpp in round 1."""
    for f in glob.glob(os.path.join(HOST, "loam_velodyne", "*.h")):
        assert "class MultiScanMapper" not in open(f).read(), f
