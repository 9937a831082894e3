"""noise::join_landmarks on the GPU (c2b_join_landmarks[_resident]) against the sequential CPU restatement of its
rule (tests/join_ref.c): the same point indices and the same counts, bit for bit, on host arrays and on the resident
problem; the errors; the preconditions; the resident chain; the reference's library property and the C++ overload."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, bits_equal
from test_gpu_bal_read import _visibility, file_vecs, from_vec_records, resident
from test_oracle_join import jn_ref  # noqa: F401  (the fixture)

pytestmark = pytest.mark.gpu

INVALID = -1
U64P, U32P, DP = ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_double)


# ---- helpers -------------------------------------------------------------------------------------------------
def raw_host(c2b, ctx, pts, off, idx, jp, seed):
    """the host-array entry on copies: (rc, point_idx after the call, stats dict)"""
    pts = np.ascontiguousarray(pts, np.float64).reshape(-1, 3)
    off = np.ascontiguousarray(off, np.uint64)
    idx = np.ascontiguousarray(idx, np.uint32).copy()
    st = c2b._lib.JoinStats()
    rc = c2b._lib.lib().c2b_join_landmarks(ctx.handle, pts.ctypes.data_as(DP), len(pts), off.ctypes.data_as(U64P),
                                           len(off) - 1, idx.ctypes.data_as(U32P), float(jp), int(seed),
                                           ctypes.byref(st))
    return rc, idx, st.to_dict()


def make_graph(rng, counts, P):
    off = np.zeros(len(counts) + 1, np.uint64)
    off[1:] = np.cumsum(counts)
    O = int(off[-1])
    return off, rng.integers(0, P, O).astype(np.uint32)


def as_problem(c2b, pts, off, idx):
    C = len(off) - 1
    cams = np.zeros((C, 15))
    cams[:, 0] = cams[:, 4] = cams[:, 8] = 1.0
    cams[:, 12] = 1.0
    return c2b.BAProblem(cams, np.asarray(pts, np.float64).reshape(-1, 3),
                         c2b.VisGraph(off, idx.astype(np.uint64), np.zeros((len(idx), 2))))


def to_resident(c2b, ctx, tmp_path, pts, off, idx):
    """the problem as the ctx's resident problem (written as .bbal, read on the GPU: points and CSR bit for bit)"""
    path = str(tmp_path / "j.bbal")
    as_problem(c2b, pts, off, idx).write_gpu(path, ctx)
    rp = resident(c2b, ctx)
    rp.read(path)
    return rp


def check_host_and_resident(c2b, ctx, jn_ref, tmp_path, pts, off, idx, jp, seed, what=""):
    ref_idx, ref_st, err = jn_ref.join_landmarks(pts, idx, jp, seed)
    assert err is None, what
    rc, got, st = raw_host(c2b, ctx, pts, off, idx, jp, seed)
    assert rc == 0, c2b._lib.lib().c2b_last_error()
    assert np.array_equal(got, ref_idx), f"{what}: host-array point indices differ ({int((got != ref_idx).sum())})"
    assert (st["n_selected"], st["n_changed"]) == (ref_st["n_selected"], ref_st["n_changed"]), what
    rp = to_resident(c2b, ctx, tmp_path, pts, off, idx)
    rst = rp.join_landmarks(jp, seed)
    assert (rst["n_selected"], rst["n_changed"]) == (ref_st["n_selected"], ref_st["n_changed"]), what
    g = rp.download()
    assert np.array_equal(g.offsets, off), what
    assert np.array_equal(g.point_idx, ref_idx), f"{what}: resident point indices differ"
    return ref_st


# ---- exactness -----------------------------------------------------------------------------------------------
def test_random_uniform(c2b, ctx, jn_ref, tmp_path):
    rng = np.random.default_rng(41)
    for t in range(6):
        P = int(rng.integers(20, 20000))
        pts = rng.uniform(-100, 100, size=(P, 3))
        counts = rng.choice([0, 1, 2, 5, 40, 300], size=int(rng.integers(1, 40)))
        off, idx = make_graph(rng, counts, P)
        for jp in (0.01, 0.3):
            check_host_and_resident(c2b, ctx, jn_ref, tmp_path, pts, off, idx, jp, 100 * t + 3, f"uniform {t} {jp}")


def test_clustered(c2b, ctx, jn_ref, tmp_path):
    """most points in a few tight clusters (many per leaf), the rest spread out"""
    rng = np.random.default_rng(42)
    centres = rng.uniform(-50, 50, size=(4, 3))
    pts = np.concatenate([centres[rng.integers(0, 4, 6000)] + rng.normal(size=(6000, 3)) * 1e-6,
                          rng.uniform(-50, 50, size=(300, 3))])
    off, idx = make_graph(rng, [700, 3, 900], len(pts))
    check_host_and_resident(c2b, ctx, jn_ref, tmp_path, pts, off, idx, 0.2, 5, "clustered")


@pytest.mark.parametrize("shape", ["planar", "collinear", "facade"])
def test_planar_and_collinear(c2b, ctx, jn_ref, tmp_path, shape):
    rng = np.random.default_rng(43)
    P = 5000
    pts = np.zeros((P, 3))
    if shape == "planar":
        pts[:, :2] = rng.uniform(-30, 30, size=(P, 2))
    elif shape == "collinear":
        pts[:, 1] = rng.uniform(-30, 30, P)
        pts[:, 0] = 2.5
    else:  # a wall on a lattice: many equal distances, ties decided by index
        pts[:, 0] = 7.0
        pts[:, 1] = (np.arange(P) % 100) * 0.25
        pts[:, 2] = (np.arange(P) // 100) * 0.25
    off, idx = make_graph(rng, [1500, 1, 1500], P)
    check_host_and_resident(c2b, ctx, jn_ref, tmp_path, pts, off, idx, 0.5, 6, shape)


def test_coincident_points(c2b, ctx, jn_ref, tmp_path):
    """groups of identical points: the (d2, index) order picks q itself for some selections"""
    rng = np.random.default_rng(44)
    base = rng.uniform(-10, 10, size=(40, 3))
    pts = base[rng.integers(0, 40, 2000)]
    off, idx = make_graph(rng, [2000, 1000], len(pts))
    st = check_host_and_resident(c2b, ctx, jn_ref, tmp_path, pts, off, idx, 1.5, 7, "coincident")
    assert st["n_selected"] == 3000 and 0 < st["n_changed"] < st["n_selected"]   # n = floor(1.5 * 2000) >= O


def test_huge_coordinates(c2b, ctx, jn_ref, tmp_path):
    """coordinates near 1e154 and above: d2 overflows to inf, the order is still (inf, index)"""
    rng = np.random.default_rng(45)
    for scale in (1e150, 1e154, 1e200, 1e300):
        pts = rng.normal(size=(300, 3)) * scale
        off, idx = make_graph(rng, [400, 200], 300)
        check_host_and_resident(c2b, ctx, jn_ref, tmp_path, pts, off, idx, 1.0, 8, f"scale {scale}")


def test_small_point_counts(c2b, ctx, jn_ref, tmp_path):
    """P = 2 ... 12: lists of m = P < 11 and m = 11 entries"""
    rng = np.random.default_rng(46)
    for P in range(2, 13):
        pts = rng.normal(size=(P, 3))
        off, idx = make_graph(rng, [30, 0, 25], P)
        st = check_host_and_resident(c2b, ctx, jn_ref, tmp_path, pts, off, idx, 100.0, P, f"P={P}")
        assert st["n_selected"] == 55 and st["n_changed"] == 55    # distinct points: never the point itself


@pytest.mark.parametrize("jp", [0.0, 1e-9, 1.0, 50.0, -1.0, float("nan")])
def test_selection_extremes(c2b, ctx, jn_ref, tmp_path, jp):
    """n >= O, n = 0 and join_percent = 0 (and negative or NaN: n = 0)"""
    rng = np.random.default_rng(47)
    pts = rng.normal(size=(500, 3))
    off, idx = make_graph(rng, [300, 0, 400], 500)
    st = check_host_and_resident(c2b, ctx, jn_ref, tmp_path, pts, off, idx, jp, 9, f"jp={jp}")
    assert st["n_selected"] == jn_ref.count(jp, 500, 700)


def test_more_selections_than_points_on_a_fresh_context(c2b, jn_ref, tmp_path):
    """k = min(floor(join_percent P), O) > P as the first join of a context: the selection scratch is sized for k,
    not only for the point sort's P entries (nothing grown by an earlier, larger call)"""
    rng = np.random.default_rng(52)
    pts = rng.uniform(-40, 40, size=(2000, 3))
    off, idx = make_graph(rng, [3000, 0, 7000], 2000)
    ref_idx, ref_st, err = jn_ref.join_landmarks(pts, idx, 3.0, 14)
    assert err is None and ref_st["n_selected"] == 6000
    for entry in ("host", "resident"):
        fresh = c2b.Context(0)
        try:
            if entry == "host":
                rc, got, st = raw_host(c2b, fresh, pts, off, idx, 3.0, 14)
                assert rc == 0, c2b._lib.lib().c2b_last_error()
            else:
                rp = to_resident(c2b, fresh, tmp_path, pts, off, idx)
                st = rp.join_landmarks(3.0, 14)
                got = rp.download().point_idx
            assert np.array_equal(got, ref_idx), entry
            assert (st["n_selected"], st["n_changed"]) == (ref_st["n_selected"], ref_st["n_changed"]), entry
            # the ctx is sound afterwards: a second call gives the same result
            rc, again, _ = raw_host(c2b, fresh, pts, off, idx, 3.0, 14)
            assert rc == 0 and np.array_equal(again, ref_idx), entry
        finally:
            fresh.close()


def test_one_long_camera(c2b, ctx, jn_ref, tmp_path):
    rng = np.random.default_rng(48)
    pts = rng.uniform(-20, 20, size=(30000, 3))
    off, idx = make_graph(rng, [5, 60000, 0, 2, 700], len(pts))
    st = check_host_and_resident(c2b, ctx, jn_ref, tmp_path, pts, off, idx, 0.5, 10, "long camera")
    assert st["n_selected"] == 15000


def test_empty(c2b, ctx, jn_ref, tmp_path):
    for off in (np.zeros(1, np.uint64), np.zeros(4, np.uint64)):
        rc, got, st = raw_host(c2b, ctx, np.ones((5, 3)), off, np.zeros(0, np.uint32), 1.0, 3)
        assert rc == 0 and len(got) == 0 and st["n_selected"] == st["n_changed"] == 0


def test_cfg2(c2b, ctx, jn_ref):
    rp, cams, pts, g = _visibility(c2b, ctx, 4, 10, 10)
    ref_idx, ref_st, err = jn_ref.join_landmarks(pts, g.point_idx, 0.1, 21)
    assert err is None and ref_st["n_changed"] > 0
    rc, got, st = raw_host(c2b, ctx, pts, g.offsets, g.point_idx, 0.1, 21)
    assert rc == 0 and np.array_equal(got, ref_idx)
    assert (st["n_selected"], st["n_changed"]) == (ref_st["n_selected"], ref_st["n_changed"])
    rst = rp.join_landmarks(0.1, 21)
    assert (rst["n_selected"], rst["n_changed"]) == (ref_st["n_selected"], ref_st["n_changed"])
    g2 = rp.download()
    assert np.array_equal(g2.point_idx, ref_idx) and np.array_equal(g2.offsets, g.offsets) and bits_equal(g2.uv, g.uv)
    edited = c2b.BAProblem(cams, pts, c2b.VisGraph(g.offsets, ref_idx.astype(np.uint64), g.uv))
    assert rp.reprojection_error(2.0) == pytest.approx(edited.total_reprojection_error(2.0), rel=1e-12)


def test_cfg3_full_size(c2b, ctx, jn_ref):
    rp, cams, pts, g = _visibility(c2b, ctx, 16, 9, 306)
    ref_idx, ref_st, err = jn_ref.join_landmarks(pts, g.point_idx, 2e-3, 22)
    assert err is None and ref_st["n_selected"] > 100
    rc, got, st = raw_host(c2b, ctx, pts, g.offsets, g.point_idx, 2e-3, 22)
    assert rc == 0 and np.array_equal(got, ref_idx)
    assert (st["n_selected"], st["n_changed"]) == (ref_st["n_selected"], ref_st["n_changed"])
    rst = rp.join_landmarks(2e-3, 22)
    assert (rst["n_selected"], rst["n_changed"]) == (ref_st["n_selected"], ref_st["n_changed"])
    assert np.array_equal(rp.download().point_idx, ref_idx)


def test_host_entry_leaves_resident_problem_alone(c2b, ctx, jn_ref):
    rp, cams, pts, g = _visibility(c2b, ctx, 4, 10, 10)
    rng = np.random.default_rng(49)
    p2 = rng.normal(size=(100, 3))
    off, idx = make_graph(rng, [3, 50, 7], 100)
    ref_idx, _, _ = jn_ref.join_landmarks(p2, idx, 0.5, 8)
    out = c2b.noise.join_landmarks_gpu(as_problem(c2b, p2, off, idx), 0.5, seed=8, ctx=ctx)
    assert np.array_equal(out.vis_graph.point_idx, ref_idx)
    after = rp.download()
    assert np.array_equal(after.point_idx, g.point_idx) and np.array_equal(after.offsets, g.offsets)


# ---- errors and preconditions --------------------------------------------------------------------------------
def test_no_neighbors(c2b, ctx, jn_ref, tmp_path):
    pts = np.ones((1, 3))
    off, idx = np.array([0, 4, 6], np.uint64), np.zeros(6, np.uint32)
    assert jn_ref.join_landmarks(pts, idx, 1.0, 1)[2] == "No neighbors?!"
    rc, got, _ = raw_host(c2b, ctx, pts, off, idx, 1.0, 1)
    assert rc == INVALID and c2b._lib.lib().c2b_last_error().decode().endswith("No neighbors?!")
    assert np.array_equal(got, idx)
    with pytest.raises(AssertionError, match="No neighbors"):
        c2b.noise.join_landmarks_gpu(as_problem(c2b, pts, off, idx), 1.0, seed=1, ctx=ctx)
    rp = to_resident(c2b, ctx, tmp_path, pts, off, idx)
    with pytest.raises(AssertionError, match="No neighbors"):
        rp.join_landmarks(1.0, 1)
    assert np.array_equal(rp.download().point_idx, idx)
    assert rp.join_landmarks(0.5, 1)["n_selected"] == 0     # n = 0: no error


@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_non_finite_point(c2b, ctx, jn_ref, tmp_path, bad):
    rng = np.random.default_rng(50)
    pts = rng.normal(size=(3000, 3))
    pts[2100, 1] = bad
    pts[2500, 0] = bad
    off, idx = make_graph(rng, [40, 60], 3000)
    assert jn_ref.join_landmarks(pts, idx, 0.01, 2)[2] == ("not finite", 2100)
    rc, got, _ = raw_host(c2b, ctx, pts, off, idx, 0.01, 2)
    assert rc == INVALID and "point 2100 " in c2b._lib.lib().c2b_last_error().decode()
    assert np.array_equal(got, idx)
    with pytest.raises(c2b.C2BError, match="not finite"):
        c2b.noise.join_landmarks_gpu(as_problem(c2b, pts, off, idx), 0.01, seed=2, ctx=ctx)
    rp = to_resident(c2b, ctx, tmp_path, pts, off, idx)
    with pytest.raises(c2b.C2BError, match="point 2100 "):
        rp.join_landmarks(0.01, 2)
    assert np.array_equal(rp.download().point_idx, idx)
    # nothing selected: no error; the ctx stays usable
    check_host_and_resident(c2b, ctx, jn_ref, tmp_path, pts, off, idx, 0.0, 2, "nothing selected")
    ok = pts.copy()
    ok[2100, 1] = ok[2500, 0] = 0.5
    check_host_and_resident(c2b, ctx, jn_ref, tmp_path, ok, off, idx, 0.01, 2, "fixed")


def test_invalid_csr(c2b, ctx):
    pts = np.random.default_rng(51).normal(size=(10, 3))
    idx = np.arange(20, dtype=np.uint32) % 10
    for off in (np.array([1, 5, 10, 15, 20], np.uint64), np.array([0, 5, 4, 15, 20], np.uint64)):
        rc, got, _ = raw_host(c2b, ctx, pts, off, idx, 1.0, 1)
        assert rc == INVALID and np.array_equal(got, idx)
    bad = idx.copy()
    bad[7] = 10
    rc, got, _ = raw_host(c2b, ctx, pts, np.array([0, 20], np.uint64), bad, 1.0, 1)
    assert rc == INVALID and np.array_equal(got, bad) and b">= 10" in c2b._lib.lib().c2b_last_error()


def test_resident_without_graph(c2b):
    from test_gpu_cull import _cfg2_inputs
    fresh = c2b.Context(0)
    try:
        st = c2b._lib.JoinStats()
        L = c2b._lib.lib()
        assert L.c2b_join_landmarks_resident(fresh.handle, 0.5, 1, ctypes.byref(st)) == INVALID
        cams, pts = _cfg2_inputs(c2b)
        rp = c2b.generate.ResidentProblem(fresh)
        rp.upload_cameras(cams)
        rp.upload_points(pts)
        assert L.c2b_join_landmarks_resident(fresh.handle, 0.5, 1, ctypes.byref(st)) == INVALID
        c2b.visibility_graph(None, cams, pts, 10.0, occlusion="analytic", ctx=fresh)
        assert L.c2b_join_landmarks_resident(fresh.handle, 0.5, 1, ctypes.byref(st)) == INVALID
        assert b"host-buffer" in L.c2b_last_error()
    finally:
        fresh.close()


# ---- the resident chain, byte for byte -------------------------------------------------------------------------
def test_resident_chain_read_join_cull_write(c2b, ctx, tmp_path):
    rp, cams, pts, g = _visibility(c2b, ctx, 4, 10, 10)
    for ext in ("bal", "bbal"):
        path = str(tmp_path / f"chain.{ext}")
        rp.write(path)
        fresh = c2b.Context(0)
        try:
            r = resident(c2b, fresh)
            r.read(path)
            st = r.join_landmarks(0.3, seed=5)
            assert st["n_changed"] > 0
            r.cull()
            out_r = str(tmp_path / f"j_r.{ext}")
            r.write(out_r)
            host = c2b.BAProblem.from_file(path)
            host.cameras = from_vec_records(c2b, file_vecs(path, host))
            h = c2b.noise.join_landmarks_gpu(host, 0.3, seed=5, ctx=fresh)
            out_h = str(tmp_path / f"j_h.{ext}")
            h.cull().write_gpu(out_h, fresh)
            assert open(out_r, "rb").read() == open(out_h, "rb").read(), f"{ext}: join + cull chain"
        finally:
            fresh.close()


# ---- the reference's library property (tests/main.rs:155-190) and the C++ overload --------------------------------
def _grid(c2b, ctx):
    from city2ba_b200 import synthetic
    return synthetic.synthetic_grid(10, 20, 3, 5., 1., 1., 1., 10., ctx=ctx)


def test_library_property(c2b, ctx):
    ba = _grid(c2b, ctx)
    out = c2b.noise.join_landmarks_gpu(ba, 0.01, seed=7, ctx=ctx)
    assert out.total_reprojection_error(2.0) > ba.total_reprojection_error(2.0)


@pytest.fixture(scope="module")
def test_join_exe(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("cpp") / "test_join")
    so_dir = os.path.join(ROOT, "city2ba_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_join.cpp"), "-o", exe, "-L", so_dir,
                           "-lcity2ba_cuda", f"-Wl,-rpath,{so_dir}"])
    return exe


def test_cpp_overload_equals_python(c2b, ctx, test_join_exe, tmp_path):
    out = str(tmp_path / "idx.u32")
    r = subprocess.run([test_join_exe, out], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "test_join ok" in r.stdout
    raw = np.fromfile(out, np.uint32)
    ba = _grid(c2b, ctx)
    O = ba.num_observations()
    assert len(raw) == 2 * O
    assert np.array_equal(raw[:O], ba.vis_graph.point_idx), "the C++ and Python grids differ"
    got = c2b.noise.join_landmarks_gpu(ba, 0.01, seed=7, ctx=ctx)
    assert np.array_equal(raw[O:], got.vis_graph.point_idx)
