"""Host side of the GPU BAL writer, without a GPU: the committed power-of-5 tables equal their generator's output,
and c2b_camera_to_vec (the camera vectors the writer formats) equals the C++ mirror's to_vec bit for bit and the
Python mirror's to_vec within 1e-13."""
import ctypes
import os
import subprocess
import sys

import numpy as np

from conftest import ROOT


def test_pow5_tables_match_generator():
    gen = os.path.join(ROOT, "city2ba_b200", "csrc", "gen_bal_tables.py")
    r = subprocess.run([sys.executable, gen, "--check"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_camera_to_vec_equals_cpp_mirror(tmp_path):
    exe = str(tmp_path / "test_bal")
    so_dir = os.path.join(ROOT, "city2ba_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_bal.cpp"), "-o", exe, "-L", so_dir,
                           "-lcity2ba_cuda", f"-Wl,-rpath,{so_dir}"])
    r = subprocess.run([exe, "--host-only"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_camera_to_vec_near_python_mirror(c2b):
    from city2ba_b200.baproblem import SnavelyCamera, from_axis_angle
    rng = np.random.default_rng(3)
    L, pd = c2b._lib.lib(), ctypes.POINTER(ctypes.c_double)
    for i in range(2000):
        a = rng.normal(size=3)
        rec = np.zeros(15)
        rec[:9] = from_axis_angle(a / np.linalg.norm(a), rng.uniform(-np.pi, np.pi) if i % 3 else np.pi)
        rec[9:] = rng.normal(size=6)
        got = np.zeros(9)
        L.c2b_camera_to_vec(rec.ctypes.data_as(pd), got.ctypes.data_as(pd))
        assert np.allclose(got, SnavelyCamera(record=rec).to_vec(), rtol=0, atol=1e-13)
