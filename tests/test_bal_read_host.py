"""The BAL reader's host part, without a GPU: c2b_camera_from_vec against the C++ mirror's SnavelyCamera::from_vec
(tests/cpp/test_bal_read.cpp, --host-only)."""
import os
import subprocess

from conftest import ROOT


def build_test_bal_read(tmp_path):
    exe = str(tmp_path / "test_bal_read")
    so_dir = os.path.join(ROOT, "city2ba_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_bal_read.cpp"), "-o", exe, "-L", so_dir,
                           "-lcity2ba_cuda", f"-Wl,-rpath,{so_dir}"])
    return exe


def test_camera_from_vec_equals_cpp_mirror(tmp_path):
    """10^5 vectors over both from_rodrigues branches, theta2 at and around 2.220446049250313e-16, bit for bit"""
    r = subprocess.run([build_test_bal_read(tmp_path), "--host-only"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
