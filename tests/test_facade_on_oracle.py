"""The header-only facade (pcl_b200/pcl_compat/pcl/**) on a machine without a GPU — CPU only.

The facade's device calls go through the C-ABI of include/pclb200.h.  Here the facade's own test programs (the same sources
tests/test_facade_gpu.py and tests/test_zz_facade_extra_gpu.py run on a B200 against libpclb200.so) are linked against a TEST
DOUBLE of that C-ABI, tests/host/pclb200_on_oracle.cpp, which answers every call with the CPU oracle.  What this proves is
the HOST side of the boundary: argument marshalling, the state the pcl:: classes keep around each call, the reference's
behaviour in the error paths, and that the expectations written into the programs are the oracle's (hence the reference's)
answers.  It proves nothing about the kernels (tests/test_traverse_host.py and the `-m gpu` tests do that), and the test
double is not a fallback: it is compiled into pytest's temporary directory and nothing in pcl_b200/ can load it."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from test_facade_gpu import FACADE, ROOT, _write_ascii_pcd, _write_binary_pcd, _write_golden

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")


@pytest.fixture(scope="module")
def double(tmp_path_factory):
    import oracle
    oracle.build()
    d = tmp_path_factory.mktemp("facade_on_oracle")
    odir = os.path.join(ROOT, "oracle")
    lib = str(d / "libpclb200_on_oracle.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wextra", "-Wno-unused-parameter",
                           "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "host", "pclb200_on_oracle.cpp"),
                           "-o", lib, "-L" + odir, "-lpcl_oracle", "-Wl,-rpath," + odir])

    def program(source):
        exe = str(d / os.path.splitext(os.path.basename(source))[0])
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-I" + FACADE, "-I" + os.path.join(ROOT, "include"),
                               os.path.join(FACADE, source), "-o", exe, lib, "-Wl,-rpath," + str(d), "-pthread"])
        return exe
    return d, lib, program


def test_the_double_exports_the_whole_c_abi(double):
    """Every entry point include/pclb200.h declares — so a facade call that is not answered fails at the call, with a
    message, instead of at link time — and none of the oracle's symbols leak into the product library."""
    import re
    _, lib, _ = double
    declared = set(re.findall(r"\b(pclb200_[a-z0-9_]+)\s*\(", open(os.path.join(ROOT, "include", "pclb200.h")).read()))
    exported = {ln.split()[-1] for ln in subprocess.check_output(["nm", "-D", "--defined-only", lib], text=True).splitlines()}
    assert declared <= exported, sorted(declared - exported)
    product = os.path.join(ROOT, "pcl_b200", "libpclb200.so")
    if os.path.exists(product):
        needed = subprocess.check_output(["readelf", "-d", product], text=True)
        assert "pcl_oracle" not in needed and "on_oracle" not in needed


def _clouds(golden, d):
    _write_ascii_pcd(d / "bun0.pcd", golden["bun0"])
    _write_binary_pcd(d / "bun4.pcd", golden["bun4"])
    return str(d / "bun0.pcd"), str(d / "bun4.pcd")


def test_reference_test_bodies_through_the_facade(double, golden, tmp_path):
    """pcl_compat/tests/test_facade.cpp: the reference's registration / kdtree / filters / features / segmentation test
    bodies written against the drop-in pcl:: classes, 8 600 checks incl. the reference's golden vectors."""
    _, _, program = double
    b0, b4 = _clouds(golden, tmp_path)
    _write_golden(tmp_path / "golden.txt", golden)
    r = subprocess.run([program("tests/test_facade.cpp"), b0, b4, str(tmp_path / "golden.txt")], capture_output=True, text=True)
    assert r.returncode == 0 and "PASSED" in r.stdout, r.stdout[-3000:] + r.stderr[-1500:]


def test_extra_facade_program(double, golden, tmp_path):
    """pcl_compat/tests/test_facade_extra.cpp: Search<PointT> overloads, CorrespondenceEstimation under a point
    representation, DefaultConvergenceCriteria thresholds, PinnedCloud, VoxelGrid leaf layout, and the host-side
    CorrespondenceRejectorSampleConsensus: the reference's golden 97 inlier pairs in order and its transform to 1e-4
    (test_registration_api.cpp:225-263), the reference's ICP with median + sample-consensus rejectors under ten random poses
    (test_registration.cpp:336-382)."""
    _, _, program = double
    b0, b4 = _clouds(golden, tmp_path)
    _write_golden(tmp_path / "golden.txt", golden)
    r = subprocess.run([program("tests/test_facade_extra.cpp"), b0, b4, str(tmp_path / "golden.txt")], capture_output=True, text=True)
    assert r.returncode == 0 and "PASSED" in r.stdout, r.stdout[-3000:] + r.stderr[-1500:]
    assert int(r.stdout.split(" checks")[0].split()[-1]) > 400   # the golden block ran


def test_icp_command_line_program(double, golden, tmp_path):
    """pcl_compat/examples/iterative_closest_point.cpp (the flow of the reference's tools/iterative_closest_point.cpp):
    blob PCD in, ICP<PointNormal, double> with injected estimators and a one-to-one rejector, concatenateFields, PCD out."""
    _, _, program = double
    b0, b4 = _clouds(golden, tmp_path)
    out = tmp_path / "aligned.pcd"
    r = subprocess.run([program("examples/iterative_closest_point.cpp"), b0, b4, str(out), "50", "0.05"], capture_output=True, text=True)
    assert r.returncode in (0, 1) and "has converged" in r.stdout, r.stdout[-2000:] + r.stderr[-1000:]
    text = out.read_text().splitlines()
    hdr = {ln.split()[0]: ln.split()[1:] for ln in text[:11] if ln and not ln.startswith("#")}
    assert hdr["FIELDS"][:3] == ["x", "y", "z"] and "normal_x" in hdr["FIELDS"] and hdr["POINTS"] == ["397"]
    body = np.array([[float(t) for t in ln.split()] for ln in text[11:] if ln.strip()])
    assert body.shape[0] == 397 and np.isfinite(body[:, :3]).all()
    tgt = np.asarray(golden["bun4"], dtype=np.float64)[:, :3]

    def mean_nn(a):
        return np.sqrt(((a[:, None, :] - tgt[None, :, :]) ** 2).sum(-1).min(1)).mean()
    assert mean_nn(body[:, :3]) < 0.5 * mean_nn(np.asarray(golden["bun0"], dtype=np.float64)[:, :3])

