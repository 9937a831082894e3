"""noise::add_incorrect_correspondences on the GPU (c2b_add_incorrect_correspondences[_resident]) against the
sequential CPU restatement of its rule (tests/mismatch_ref.c): the same point indices and the same
counts, bit for bit, on host arrays and on the resident problem; the errors of Rng::weighted; the resident chains."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, bits_equal
from test_gpu_bal_read import _visibility, file_vecs, from_vec_records, resident
from test_oracle_mismatch import mm_ref  # noqa: F401  (the fixture)

pytestmark = pytest.mark.gpu

INVALID = -1
U64P, U32P, DP = ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_double)


# ---- helpers -------------------------------------------------------------------------------------------------
def raw_host(c2b, ctx, off, idx, uv, p, seed):
    """the host-array entry on copies: (rc, point_idx after the call, stats dict)"""
    off = np.ascontiguousarray(off, np.uint64)
    idx = np.ascontiguousarray(idx, np.uint32).copy()
    uv = np.ascontiguousarray(uv, np.float64).reshape(-1, 2)
    st = c2b._lib.MismatchStats()
    rc = c2b._lib.lib().c2b_add_incorrect_correspondences(ctx.handle, off.ctypes.data_as(U64P), len(off) - 1,
                                                          idx.ctypes.data_as(U32P), uv.ctypes.data_as(DP), float(p),
                                                          int(seed), ctypes.byref(st))
    return rc, idx, st.to_dict()


def make_graph(rng, counts, P=1000):
    off = np.zeros(len(counts) + 1, np.uint64)
    off[1:] = np.cumsum(counts)
    O = int(off[-1])
    return off, rng.integers(0, P, O).astype(np.uint32), rng.normal(size=(O, 2)) * 100.0


def as_problem(c2b, off, idx, uv, P=1000):
    C = len(off) - 1
    cams = np.zeros((C, 15))
    cams[:, 0] = cams[:, 4] = cams[:, 8] = 1.0
    cams[:, 12] = 1.0
    return c2b.BAProblem(cams, np.zeros((P, 3)), c2b.VisGraph(off, idx.astype(np.uint64), uv))


def to_resident(c2b, ctx, tmp_path, off, idx, uv, P=1000):
    """the graph as the ctx's resident problem (written as .bbal, read on the GPU: the CSR bit for bit)"""
    path = str(tmp_path / "g.bbal")
    as_problem(c2b, off, idx, uv, P).write_gpu(path, ctx)
    rp = resident(c2b, ctx)
    rp.read(path)
    return rp


def check_host_and_resident(c2b, ctx, mm_ref, tmp_path, off, idx, uv, p, seed, what=""):
    ref_idx, ref_st, err = mm_ref.add_incorrect_correspondences(off, idx, uv, p, seed)
    assert err is None, what
    rc, got, st = raw_host(c2b, ctx, off, idx, uv, p, seed)
    assert rc == 0, c2b._lib.lib().c2b_last_error()
    assert np.array_equal(got, ref_idx), f"{what}: host-array point indices differ"
    assert (st["n_selected"], st["n_swapped"]) == (ref_st["n_selected"], ref_st["n_swapped"]), what
    rp = to_resident(c2b, ctx, tmp_path, off, idx, uv)
    rst = rp.add_incorrect_correspondences(p, seed)
    assert (rst["n_selected"], rst["n_swapped"]) == (ref_st["n_selected"], ref_st["n_swapped"]), what
    g = rp.download()
    assert np.array_equal(g.offsets, off) and bits_equal(g.uv, uv), what
    assert np.array_equal(g.point_idx, ref_idx), f"{what}: resident point indices differ"
    return ref_st


# ---- exactness -----------------------------------------------------------------------------------------------
def test_random_graphs(c2b, ctx, mm_ref, tmp_path):
    """cameras of 0, 1, 2 and many observations, duplicated (u, v) within a camera"""
    rng = np.random.default_rng(31)
    for t in range(12):
        counts = rng.choice([0, 1, 2, 3, 17, 40, 300], size=int(rng.integers(1, 60)))
        off, idx, uv = make_graph(rng, counts)
        if len(uv) > 4:
            uv[rng.integers(0, len(uv), 3)] = uv[0]
        for p in (0.3, 1.0):
            check_host_and_resident(c2b, ctx, mm_ref, tmp_path, off, idx, uv, p, 1000 * t + 7, f"random {t} p={p}")


def test_one_long_camera(c2b, ctx, mm_ref, tmp_path):
    """one camera of 40,000 observations, far longer than any tile, beside short ones"""
    rng = np.random.default_rng(32)
    off, idx, uv = make_graph(rng, [5, 40000, 0, 2, 700])
    st = check_host_and_resident(c2b, ctx, mm_ref, tmp_path, off, idx, uv, 0.05, 99, "long camera")
    assert st["n_selected"] > 1500 and st["n_swapped"] > 1500


@pytest.mark.parametrize("p", [0.0, 1.0, float("nan")])
def test_chance_extremes(c2b, ctx, mm_ref, tmp_path, p):
    rng = np.random.default_rng(33)
    counts = np.array([0, 1, 2, 9, 50, 1, 30])
    off, idx, uv = make_graph(rng, counts)
    st = check_host_and_resident(c2b, ctx, mm_ref, tmp_path, off, idx, uv, p, 5, f"p={p}")
    assert st["n_selected"] == (int(counts[counts > 1].sum()) if p == 1.0 else 0)


def test_empty(c2b, ctx, mm_ref, tmp_path):
    for off in (np.zeros(1, np.uint64), np.zeros(4, np.uint64)):
        rc, got, st = raw_host(c2b, ctx, off, np.zeros(0, np.uint32), np.zeros((0, 2)), 1.0, 3)
        assert rc == 0 and len(got) == 0 and st["n_selected"] == st["n_swapped"] == 0
    rp = to_resident(c2b, ctx, tmp_path, np.zeros(4, np.uint64), np.zeros(0, np.uint32), np.zeros((0, 2)))
    st = rp.add_incorrect_correspondences(1.0, 3)
    assert st["n_selected"] == st["n_swapped"] == 0 and rp.download().num_observations == 0


def test_cfg2(c2b, ctx, mm_ref, tmp_path):
    rp, cams, pts, g = _visibility(c2b, ctx, 4, 10, 10)
    ref_idx, ref_st, err = mm_ref.add_incorrect_correspondences(g.offsets, g.point_idx, g.uv, 0.1, 21)
    assert err is None and ref_st["n_swapped"] > 0
    rc, got, st = raw_host(c2b, ctx, g.offsets, g.point_idx, g.uv, 0.1, 21)
    assert rc == 0 and np.array_equal(got, ref_idx)
    assert (st["n_selected"], st["n_swapped"]) == (ref_st["n_selected"], ref_st["n_swapped"])
    rst = rp.add_incorrect_correspondences(0.1, 21)
    assert (rst["n_selected"], rst["n_swapped"]) == (ref_st["n_selected"], ref_st["n_swapped"])
    g2 = rp.download()
    assert np.array_equal(g2.point_idx, ref_idx) and np.array_equal(g2.offsets, g.offsets) and bits_equal(g2.uv, g.uv)
    # the resident reprojection error sees the edited graph
    edited = c2b.BAProblem(cams, pts, c2b.VisGraph(g.offsets, ref_idx.astype(np.uint64), g.uv))
    assert rp.reprojection_error(2.0) == pytest.approx(edited.total_reprojection_error(2.0), rel=1e-12)
    assert rp.reprojection_error(2.0) > c2b.BAProblem(cams, pts, g).total_reprojection_error(2.0)


def test_cfg3_full_size(c2b, ctx, mm_ref):
    rp, cams, pts, g = _visibility(c2b, ctx, 16, 9, 306)
    ref_idx, ref_st, err = mm_ref.add_incorrect_correspondences(g.offsets, g.point_idx, g.uv, 0.01, 22)
    assert err is None
    rc, got, st = raw_host(c2b, ctx, g.offsets, g.point_idx, g.uv, 0.01, 22)
    assert rc == 0 and np.array_equal(got, ref_idx)
    assert (st["n_selected"], st["n_swapped"]) == (ref_st["n_selected"], ref_st["n_swapped"])
    rst = rp.add_incorrect_correspondences(0.01, 22)
    assert (rst["n_selected"], rst["n_swapped"]) == (ref_st["n_selected"], ref_st["n_swapped"])
    assert np.array_equal(rp.download().point_idx, ref_idx)


def test_host_entry_leaves_resident_problem_alone(c2b, ctx, mm_ref, tmp_path):
    rp, cams, pts, g = _visibility(c2b, ctx, 4, 10, 10)
    rng = np.random.default_rng(34)
    off, idx, uv = make_graph(rng, [3, 50, 7])
    ref_idx, _, _ = mm_ref.add_incorrect_correspondences(off, idx, uv, 0.5, 8)
    out = c2b.noise.add_incorrect_correspondences_gpu(as_problem(c2b, off, idx, uv), 0.5, seed=8, ctx=ctx)
    assert np.array_equal(out.vis_graph.point_idx, ref_idx)
    after = rp.download()
    assert np.array_equal(after.point_idx, g.point_idx) and np.array_equal(after.offsets, g.offsets)
    assert bits_equal(after.uv, g.uv)


# ---- errors --------------------------------------------------------------------------------------------------
def _bad_graph(kind):
    rng = np.random.default_rng(35)
    off, idx, uv = make_graph(rng, [4, 1, 6, 5])
    uv[4] = np.nan   # camera 1 has one observation: never drawn from
    if kind == "AllWeightsZero":
        uv[11:16] = uv[11]      # camera 3: every observation at the same (u, v)
    else:
        uv[8] = (np.inf, 0.0)   # camera 2
    return off, idx, uv


@pytest.mark.parametrize("kind", ["AllWeightsZero", "NegativeWeight"])
def test_weight_errors(c2b, ctx, mm_ref, tmp_path, kind):
    off, idx, uv = _bad_graph(kind)
    _, _, err = mm_ref.add_incorrect_correspondences(off, idx, uv, 1.0, 4)
    assert err[0] == kind
    tail = f"called `Result::unwrap()` on an `Err` value: {kind}"
    rc, got, _ = raw_host(c2b, ctx, off, idx, uv, 1.0, 4)
    msg = c2b._lib.lib().c2b_last_error().decode()
    assert rc == INVALID and msg.endswith(tail) and f"CSR index {err[1]})" in msg
    assert np.array_equal(got, idx)
    with pytest.raises(AssertionError, match=kind):
        c2b.noise.add_incorrect_correspondences_gpu(as_problem(c2b, off, idx, uv), 1.0, seed=4, ctx=ctx)
    rp = to_resident(c2b, ctx, tmp_path, off, idx, uv)
    with pytest.raises(AssertionError, match=kind):
        rp.add_incorrect_correspondences(1.0, 4)
    g = rp.download()
    assert np.array_equal(g.point_idx, idx) and bits_equal(g.uv, uv)
    # nothing selected in the failing camera: no error
    check_host_and_resident(c2b, ctx, mm_ref, tmp_path, off, idx, uv, 0.0, 4, "nothing selected")
    ok = uv.copy()
    ok[8:] = np.random.default_rng(1).normal(size=(len(uv) - 8, 2))
    check_host_and_resident(c2b, ctx, mm_ref, tmp_path, off, idx, ok, 1.0, 4, "fixed")
    # the ctx stays usable: a valid call equals one on a fresh ctx
    rng = np.random.default_rng(36)
    off2, idx2, uv2 = make_graph(rng, [30, 2, 500])
    _, a, sa = raw_host(c2b, ctx, off2, idx2, uv2, 0.4, 12)
    fresh = c2b.Context(0)
    try:
        _, b, sb = raw_host(c2b, fresh, off2, idx2, uv2, 0.4, 12)
    finally:
        fresh.close()
    assert np.array_equal(a, b) and (sa["n_selected"], sa["n_swapped"]) == (sb["n_selected"], sb["n_swapped"])
    rst = rp.add_incorrect_correspondences(0.0, 4)   # the resident problem is still there
    assert rst["n_selected"] == 0


@pytest.mark.parametrize("bad", ["first_offset", "decreasing"])
def test_invalid_offsets(c2b, ctx, bad):
    rng = np.random.default_rng(37)
    off = np.array([0, 5, 10, 15, 20], np.uint64)
    idx = rng.integers(0, 6, 20).astype(np.uint32)
    uv = rng.normal(size=(20, 2))
    if bad == "first_offset":
        off[0] = 1
    else:
        off[2] = 4
    rc, got, _ = raw_host(c2b, ctx, off, idx, uv, 1.0, 1)
    assert rc == INVALID and np.array_equal(got, idx)


def test_resident_without_result(c2b):
    from test_gpu_cull import _cfg2_inputs
    fresh = c2b.Context(0)
    try:
        st = c2b._lib.MismatchStats()
        L = c2b._lib.lib()
        assert L.c2b_add_incorrect_correspondences_resident(fresh.handle, 0.5, 1, ctypes.byref(st)) == INVALID
        cams, pts = _cfg2_inputs(c2b)
        rp = c2b.generate.ResidentProblem(fresh)
        rp.upload_cameras(cams)
        rp.upload_points(pts)
        assert L.c2b_add_incorrect_correspondences_resident(fresh.handle, 0.5, 1, ctypes.byref(st)) == INVALID
        c2b.visibility_graph(None, cams, pts, 10.0, occlusion="analytic", ctx=fresh)
        assert L.c2b_add_incorrect_correspondences_resident(fresh.handle, 0.5, 1, ctypes.byref(st)) == INVALID
        assert b"host-buffer" in L.c2b_last_error()
    finally:
        fresh.close()


# ---- the resident chains, byte for byte ------------------------------------------------------------------------
def _host_from_file(c2b, path):
    host = c2b.BAProblem.from_file(path)
    host.cameras = from_vec_records(c2b, file_vecs(path, host))   # the C++ mirror's from_vec, as the reader's
    return host


def _chain(c2b, ctx, tmp_path, n, cpb, ppb, what):
    from city2ba_b200 import noise
    rp, cams, pts, g = _visibility(c2b, ctx, n, cpb, ppb)
    for ext in ("bal", "bbal"):
        path = str(tmp_path / f"chain.{ext}")
        rp.write(path)
        fresh = c2b.Context(0)
        try:
            r = resident(c2b, fresh)
            # read -> drift -> noise -> mismatch -> write
            r.read(path)
            r.add_drift(0.01, 0.001, 0.1, seed=3)
            r.add_noise(0.01, 0.001, 0.01, 0.001, seed=4)
            st = r.add_incorrect_correspondences(0.05, seed=5)
            assert st["n_swapped"] > 0
            out_r = str(tmp_path / f"mm_r.{ext}")
            r.write(out_r)
            h = noise.add_drift_normalized(_host_from_file(c2b, path), 0.01, 0.001, 0.1, seed=3, ctx=fresh)
            h = noise.add_noise(h, 0.01, 0.001, 0.01, 0.001, seed=4, ctx=fresh)
            h = noise.add_incorrect_correspondences_gpu(h, 0.05, seed=5, ctx=fresh)
            out_h = str(tmp_path / f"mm_h.{ext}")
            h.write_gpu(out_h, fresh)
            assert open(out_r, "rb").read() == open(out_h, "rb").read(), f"{what} {ext}: noise + mismatch chain"
            # read -> mismatch -> cull -> write (point indices no longer ascend within a camera)
            r.read(path)
            r.add_incorrect_correspondences(0.2, seed=6)
            r.cull()
            out_c = str(tmp_path / f"mmc_r.{ext}")
            r.write(out_c)
            hm = noise.add_incorrect_correspondences_gpu(_host_from_file(c2b, path), 0.2, seed=6, ctx=fresh)
            o = hm.vis_graph.offsets.astype(np.int64)
            assert any(np.any(np.diff(hm.vis_graph.point_idx[o[c]:o[c + 1]].astype(np.int64)) < 0)
                       for c in range(len(o) - 1))
            out_hc = str(tmp_path / f"mmc_h.{ext}")
            hm.cull().write_gpu(out_hc, fresh)
            assert open(out_c, "rb").read() == open(out_hc, "rb").read(), f"{what} {ext}: mismatch + cull chain"
        finally:
            fresh.close()


def test_resident_chain_cfg2(c2b, ctx, tmp_path):
    _chain(c2b, ctx, tmp_path, 4, 10, 10, "cfg2")


def test_resident_chain_cfg3_full_size(c2b, ctx, tmp_path):
    _chain(c2b, ctx, tmp_path, 16, 9, 306, "cfg3")


# ---- the reference's library property (tests/main.rs:155-190) and the C++ overload --------------------------------
def _grid(c2b, ctx):
    from city2ba_b200 import synthetic
    return synthetic.synthetic_grid(10, 20, 3, 5., 1., 1., 1., 10., ctx=ctx)


def test_library_property(c2b, ctx):
    ba = _grid(c2b, ctx)
    out = c2b.noise.add_incorrect_correspondences_gpu(ba, 0.01, seed=4, ctx=ctx)
    assert out.total_reprojection_error(2.0) > ba.total_reprojection_error(2.0)


@pytest.fixture(scope="module")
def test_mismatch_exe(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("cpp") / "test_mismatch")
    so_dir = os.path.join(ROOT, "city2ba_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_mismatch.cpp"), "-o", exe, "-L", so_dir,
                           "-lcity2ba_cuda", f"-Wl,-rpath,{so_dir}"])
    return exe


def test_cpp_overload_equals_python(c2b, ctx, test_mismatch_exe, tmp_path):
    out = str(tmp_path / "idx.u32")
    r = subprocess.run([test_mismatch_exe, out], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "test_mismatch ok" in r.stdout
    raw = np.fromfile(out, np.uint32)
    ba = _grid(c2b, ctx)
    O = ba.num_observations()
    assert len(raw) == 2 * O
    assert np.array_equal(raw[:O], ba.vis_graph.point_idx), "the C++ and Python grids differ"
    got = c2b.noise.add_incorrect_correspondences_gpu(ba, 0.01, seed=4, ctx=ctx)
    assert np.array_equal(raw[O:], got.vis_graph.point_idx)
    assert not math.isnan(got.total_reprojection_error(2.0))
