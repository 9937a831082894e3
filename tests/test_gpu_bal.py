"""BAL files written on the GPU (c2b_write_bal / c2b_write_bal_resident) against an independent number oracle and
the host writers of both mirrors.

The oracle for one f64 is Python's shortest round-trip repr, expanded to positional notation by Decimal, with a
trailing ".0" / zeros trimmed, and "NaN" / "inf" / "-inf": the spelling of Rust's `{}` (src/baproblem.rs:709-733).
It shares no code with the GPU encoder or either mirror."""
import ctypes
import math
import os
import struct
import subprocess
from decimal import Decimal

import numpy as np
import pytest

from conftest import ROOT, bits_equal

pytestmark = pytest.mark.gpu

INVALID, IO = -1, -7


def oracle(x: float) -> str:
    if math.isnan(x):
        return "NaN"
    if math.isinf(x):
        return "inf" if x > 0 else "-inf"
    r = repr(x)
    if "e" not in r:  # repr is already positional: only the ".0" of integers goes
        return r[:-2] if r.endswith(".0") else r
    s = format(Decimal(r), "f")
    return s.rstrip("0").rstrip(".") if "." in s else s


def special_values():
    d = lambda bits: struct.unpack("<d", struct.pack("<Q", bits))[0]  # noqa: E731
    v = [0.0, 5e-324, d((1 << 52) - 1), 2.2250738585072014e-308, 1.7976931348623157e308, math.nan, math.inf,
         1.0, 0.1, 0.3, 0.1 + 0.2, 1e21, 1e22, 1e23, 2.0 ** 60, 123456789012345680000.0, 1 / 3, math.pi]
    for e in range(-1074, 1024):  # powers of two and their neighbours
        p = math.ldexp(1.0, e)
        v += [p, float(np.nextafter(p, 0.0)), float(np.nextafter(p, math.inf))]
    for e in range(-323, 309):  # powers of ten and their neighbours
        p = float(f"1e{e}")
        v += [p, float(np.nextafter(p, 0.0)), float(np.nextafter(p, math.inf))]
    v += [d(e << 52) for e in range(1, 2047)]  # mantissa 0: the asymmetric interval
    v += [float(2 ** 53 + k) for k in range(-300, 300)]
    for p in range(15, 24):
        v += [float(10 ** p + k * 10 ** max(0, p - 16)) for k in range(-50, 50)]
    v += [0.1 * k for k in range(1, 1000)] + [d(0x3FF0000000000000 + k) for k in range(1, 1000)]  # 17 digits
    a = np.array(v, np.float64)
    return np.concatenate([a, -a])  # -0.0 among them


def points_only(c2b, vals):
    """a problem with C = 0, O = 0 and the values as P x 3 coordinates (padded with zeros)"""
    vals = np.concatenate([vals, np.zeros((-len(vals)) % 3)])
    g = c2b.VisGraph(np.zeros(1, np.uint64), np.zeros(0, np.uint64), np.zeros((0, 2)))
    return c2b.BAProblem(np.zeros((0, 15)), vals.reshape(-1, 3), g), vals


def check_numbers(c2b, ctx, vals, path):
    ba, vals = points_only(c2b, vals)
    ba.write_gpu(path, ctx)
    data = open(path, "rb").read().decode()
    lines = data.split("\n")
    assert lines[0] == f"0 {len(ba.points)} 0" and lines[-1] == ""
    toks = " ".join(lines[1:-1]).split(" ")
    assert len(toks) == len(vals)
    exp = [oracle(x) for x in vals.tolist()]
    if toks != exp:
        bad = [(x, t, e) for x, t, e in zip(vals.tolist(), toks, exp) if t != e]
        pytest.fail(f"{len(bad)} values differ from the oracle, e.g. {bad[:3]}")
    back = np.array(toks, np.float64)
    nan = np.isnan(vals)
    assert np.array_equal(np.isnan(back), nan)
    assert bits_equal(back[~nan], vals[~nan]), "a GPU string does not parse back to the same double"


def test_numbers_special(c2b, ctx, tmp_path):
    v = special_values()
    v = np.concatenate([v, [-math.nan, -math.inf, struct.unpack("<d", struct.pack("<Q", 0xFFF8000000000001))[0]]])
    check_numbers(c2b, ctx, v, str(tmp_path / "special.bal"))


@pytest.mark.parametrize("kind", ["bits", "unit", "thousand"])
def test_numbers_random(c2b, ctx, tmp_path, kind):
    """10^7 values of each kind, in batches of 10^6"""
    rng = np.random.default_rng({"bits": 1, "unit": 2, "thousand": 3}[kind])
    for b in range(10):
        if kind == "bits":
            v = rng.integers(0, 2 ** 64, 10 ** 6, dtype=np.uint64).view(np.float64)
        elif kind == "unit":
            v = rng.uniform(-1.0, 1.0, 10 ** 6)
        else:
            v = rng.uniform(-1000.0, 1000.0, 10 ** 6)
        check_numbers(c2b, ctx, v, str(tmp_path / f"{kind}{b}.bal"))


# ---- whole files ---------------------------------------------------------------------------------------------------
def camera_vecs(c2b, cams):
    """c2b_camera_to_vec of every record (the vectors the GPU writer formats)"""
    L, pd = c2b._lib.lib(), ctypes.POINTER(ctypes.c_double)
    out = np.zeros((len(cams), 9))
    for i, c in enumerate(np.ascontiguousarray(cams, np.float64)):
        L.c2b_camera_to_vec(c.ctypes.data_as(pd), out[i].ctypes.data_as(pd))
    return out


def random_problem(c2b, rng, C, P, max_obs, empty_every=0):
    from city2ba_b200.baproblem import from_axis_angle
    cams = np.zeros((C, 15))
    for i in range(C):
        a = rng.normal(size=3)
        cams[i, :9] = from_axis_angle(a / np.linalg.norm(a), rng.uniform(-3.1, 3.1))
        cams[i, 9:] = rng.normal(size=6) * 10.0 ** rng.integers(-3, 4, 6)
    pts = rng.normal(size=(P, 3)) * 10.0 ** rng.integers(-5, 6, (P, 1))
    counts = rng.integers(0, max_obs + 1, C) if P else np.zeros(C, np.int64)
    if empty_every:
        counts[::empty_every] = 0
    off = np.zeros(C + 1, np.uint64)
    off[1:] = np.cumsum(counts)
    O = int(off[-1])
    idx = rng.integers(0, max(P, 1), O).astype(np.uint64)
    uv = rng.normal(size=(O, 2))
    uv[rng.random(O) < 0.05] *= -0.0
    return c2b.BAProblem(cams, pts, c2b.VisGraph(off, idx, uv))


def split_text(data, ba):
    """(header + observation lines, camera lines, point lines) of a text BAL file"""
    lines = data.split(b"\n")
    O, C = ba.num_observations(), ba.num_cameras()
    return lines[:1 + O], lines[1 + O:1 + O + C], lines[1 + O + C:]


def camera_block(ba):
    """byte range of the camera 9-vectors in a binary BAL file"""
    start = 24 + 8 * ba.num_cameras() + 24 * ba.num_observations()
    return start, start + 72 * ba.num_cameras()


def assert_matches_mirrors(c2b, ba, gpu_text, gpu_bin, tmp_path, what=""):
    """text: header / observation / point lines equal Python's write_text (all values finite), camera lines are
    the oracle's spelling of c2b_camera_to_vec; binary: equal to Python's write_binary outside the camera block,
    the block equal to c2b_camera_to_vec's bits and to Python's to_vec within 1e-13.  Returns whether Python's
    camera block is bit-equal."""
    ref_t, ref_b = str(tmp_path / "ref.bal"), str(tmp_path / "ref.bbal")
    ba.write_text(ref_t)
    ba.write_binary(ref_b)
    a, b = open(ref_t, "rb").read(), gpu_text
    ha, ca, pa = split_text(a, ba)
    hb, cb, pb = split_text(b, ba)
    assert ha == hb, f"{what}: header or observation lines differ from write_text"
    assert pa == pb, f"{what}: point lines differ from write_text"
    vecs = camera_vecs(c2b, ba.cameras)
    assert cb == [" ".join(oracle(x) for x in v).encode() for v in vecs.tolist()], f"{what}: camera lines"
    ra = open(ref_b, "rb").read()
    s, e = camera_block(ba)
    assert len(ra) == len(gpu_bin) and ra[:s] == gpu_bin[:s] and ra[e:] == gpu_bin[e:], f"{what}: binary differs"
    got = np.frombuffer(gpu_bin[s:e], ">f8").reshape(-1, 9)
    assert bits_equal(got.astype(np.float64), vecs), f"{what}: binary camera block"
    py = np.frombuffer(ra[s:e], ">f8").reshape(-1, 9).astype(np.float64)
    assert np.allclose(got, py, rtol=0, atol=1e-13), f"{what}: camera block vs Python's to_vec"
    return ra[s:e] == gpu_bin[s:e]


def gpu_files(c2b, ctx, ba, tmp_path, name="gpu"):
    t, b = str(tmp_path / f"{name}.bal"), str(tmp_path / f"{name}.bbal")
    st_t, st_b = {}, {}
    ba.write_gpu(t, ctx, stats=st_t)
    ba.write_gpu(b, ctx, stats=st_b)
    dt, db = open(t, "rb").read(), open(b, "rb").read()
    assert st_t["bytes"] == len(dt) and st_b["bytes"] == len(db)
    return dt, db


def test_whole_files_random(c2b, ctx, tmp_path):
    rng = np.random.default_rng(5)
    equal = []
    for C, P, k in [(1, 1, 3), (7, 40, 9), (60, 800, 50), (400, 20000, 300)]:
        ba = random_problem(c2b, rng, C, P, k, empty_every=5)
        dt, db = gpu_files(c2b, ctx, ba, tmp_path)
        equal.append(assert_matches_mirrors(c2b, ba, dt, db, tmp_path, f"C={C}"))
    print(f"binary camera block bit-equal to Python's to_vec: {equal}")


@pytest.mark.parametrize("case", ["empty", "cameras_no_obs", "empty_cameras", "points_only"])
def test_edge_problems(c2b, ctx, tmp_path, case):
    rng = np.random.default_rng(6)
    ba = {"empty": lambda: random_problem(c2b, rng, 0, 0, 0),
          "cameras_no_obs": lambda: random_problem(c2b, rng, 6, 10, 0),
          "empty_cameras": lambda: random_problem(c2b, rng, 30, 50, 8, empty_every=2),
          "points_only": lambda: random_problem(c2b, rng, 0, 25, 0)}[case]()
    dt, db = gpu_files(c2b, ctx, ba, tmp_path)
    assert_matches_mirrors(c2b, ba, dt, db, tmp_path, case)
    if case == "empty":
        assert dt == b"0 0 0\n" and db == bytes(24)


# ---- chunking ------------------------------------------------------------------------------------------------------
def test_chunk_boundaries(c2b, ctx, tmp_path):
    """small chunks cut inside runs of 326-byte values and at camera boundaries: the same bytes as one chunk, and
    the same bytes on a second call"""
    rng = np.random.default_rng(8)
    ba = random_problem(c2b, rng, 40, 3000, 30, empty_every=3)
    sub = np.array([5e-324, -5e-324, 2.2250738585072009e-308, -1.5e-323])
    ba.points[::7] = rng.choice(sub, size=ba.points[::7].shape)
    ba.vis_graph.uv[::5] = rng.choice(sub, size=ba.vis_graph.uv[::5].shape)
    ref_t, ref_b = gpu_files(c2b, ctx, ba, tmp_path, "default")
    try:
        for chunk in (4096, 4096 + 8, 5000, 65536):
            ctx.tune("bal_chunk_bytes", chunk)
            for rep in range(2):
                dt, db = gpu_files(c2b, ctx, ba, tmp_path, f"c{chunk}_{rep}")
                assert dt == ref_t and db == ref_b, f"chunk {chunk}, call {rep}"
            st = {}
            ba.write_gpu(str(tmp_path / "stats.bal"), ctx, stats=st)
            assert st["chunks"] >= len(ref_t) // chunk
    finally:
        ctx.tune("reset", 0)
    assert_matches_mirrors(c2b, ba, ref_t, ref_b, tmp_path, "subnormal runs")


# ---- the resident chain ----------------------------------------------------------------------------------------------
def _resident(c2b, ctx, cams, pts, scene, **kw):
    rp = c2b.generate.ResidentProblem(ctx)
    rp.upload_cameras(cams)
    rp.upload_points(pts)
    rp.run(scene, 10.0, **kw)
    return rp


def _chain(c2b, ctx, rp, tmp_path, what):
    """cull, drift, noise, then the resident write against download + host-array GPU writer + mirrors"""
    st = rp.cull()
    rp.add_drift(0.01, 0.001, 0.1, seed=3)
    rp.add_noise(0.01, 0.001, 0.01, 0.001, seed=4)
    files = {}
    for ext in ("bal", "bbal"):
        p = str(tmp_path / f"resident.{ext}")
        s = rp.write(p)
        files[ext] = open(p, "rb").read()
        assert s["bytes"] == len(files[ext])
    c, p = rp.download_problem(st["n_cameras"], st["n_points"])
    ba = c2b.BAProblem(c, p, rp.download())
    assert ba.num_observations() > 0, what
    dt, db = gpu_files(c2b, ctx, ba, tmp_path, "host_entry")
    assert dt == files["bal"] and db == files["bbal"], f"{what}: resident and host-array entries differ"
    assert_matches_mirrors(c2b, ba, dt, db, tmp_path, what)


def test_resident_chain_cfg2(c2b, ctx, tmp_path):
    from city2ba_b200 import synthetic
    cams = synthetic.grid_cameras(10, 4, 20.0, 1.0)
    pts = synthetic.grid_points(10, 4, 20.0, 1.0, 1.0)
    xyz, tri = synthetic.city_mesh(4)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    _chain(c2b, ctx, _resident(c2b, ctx, cams, pts, scene), tmp_path, "cfg2")


def test_resident_chain_cfg3_full_size(c2b, ctx, tmp_path):
    from city2ba_b200 import synthetic
    cams = synthetic.grid_cameras(9, 16, 20.0, 1.0)
    pts = synthetic.grid_points(306, 16, 20.0, 1.0, 1.0)
    xyz, tri = synthetic.city_mesh(16)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    _chain(c2b, ctx, _resident(c2b, ctx, cams, pts, scene), tmp_path, "cfg3")


def test_host_entry_leaves_resident_problem_alone(c2b, ctx, tmp_path):
    from city2ba_b200 import synthetic
    cams = synthetic.grid_cameras(10, 4, 20.0, 1.0)
    pts = synthetic.grid_points(10, 4, 20.0, 1.0, 1.0)
    rp = _resident(c2b, ctx, cams, pts, None, occlusion="analytic")
    before = rp.download()
    cb, pb = rp.download_problem(len(cams), len(pts))
    first = rp.write(str(tmp_path / "a.bal"))
    rng = np.random.default_rng(9)
    for _ in range(3):
        random_problem(c2b, rng, 50, 400, 30).write_gpu(str(tmp_path / "other.bal"), ctx)
    after = rp.download()
    ca, pa = rp.download_problem(len(cams), len(pts))
    assert np.array_equal(before.offsets, after.offsets) and np.array_equal(before.point_idx, after.point_idx)
    assert bits_equal(before.uv, after.uv) and bits_equal(cb, ca) and bits_equal(pb, pa)
    again = rp.write(str(tmp_path / "b.bal"))
    assert first["bytes"] == again["bytes"]
    assert open(tmp_path / "a.bal", "rb").read() == open(tmp_path / "b.bal", "rb").read()


# ---- errors --------------------------------------------------------------------------------------------------------
def test_unwritable_path(c2b, ctx, tmp_path):
    from city2ba_b200.baproblem import IOError_
    ba = random_problem(c2b, np.random.default_rng(1), 3, 5, 4)
    for ext in ("bal", "bbal"):
        with pytest.raises(IOError_):
            ba.write_gpu(str(tmp_path / "missing" / f"x.{ext}"), ctx)
    with pytest.raises(IOError_):
        ba.write_gpu(str(tmp_path / "x.txt"), ctx)  # the mirrors' extension dispatch


@pytest.mark.parametrize("bad", ["first_offset", "decreasing", "index_range"])
def test_invalid_csr_creates_no_file(c2b, ctx, tmp_path, bad):
    rng = np.random.default_rng(13)
    cams, pts = rng.normal(size=(4, 15)), rng.normal(size=(6, 3))
    off = np.array([0, 5, 10, 15, 20], np.uint64)
    idx = rng.integers(0, 6, 20).astype(np.uint32)
    uv = rng.normal(size=(20, 2))
    if bad == "first_offset":
        off[0] = 1
    elif bad == "decreasing":
        off[2] = 4
    else:
        idx[17] = 6
    path = str(tmp_path / "bad.bal")
    pd = ctypes.POINTER(ctypes.c_double)
    rc = c2b._lib.lib().c2b_write_bal(ctx.handle, path.encode(), 0, cams.ctypes.data_as(pd), 4, pts.ctypes.data_as(pd),
                                      6, off.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)),
                                      idx.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), uv.ctypes.data_as(pd),
                                      None)
    assert rc == INVALID and not os.path.exists(path)


def test_resident_write_without_result(c2b, tmp_path):
    fresh = c2b.Context(0)
    try:
        path = str(tmp_path / "r.bal")
        assert c2b._lib.lib().c2b_write_bal_resident(fresh.handle, path.encode(), 0, None) == INVALID
        from city2ba_b200 import synthetic
        rp = c2b.generate.ResidentProblem(fresh)
        rp.upload_cameras(synthetic.grid_cameras(10, 4, 20.0, 1.0))
        rp.upload_points(synthetic.grid_points(10, 4, 20.0, 1.0, 1.0))
        assert c2b._lib.lib().c2b_write_bal_resident(fresh.handle, path.encode(), 0, None) == INVALID
        assert not os.path.exists(path)
    finally:
        fresh.close()


def test_resident_write_after_host_buffer_call(c2b, tmp_path):
    from city2ba_b200 import synthetic
    fresh = c2b.Context(0)
    try:
        cams = synthetic.grid_cameras(10, 4, 20.0, 1.0)
        pts = synthetic.grid_points(10, 4, 20.0, 1.0, 1.0)
        c2b.visibility_graph(None, cams, pts, 10.0, occlusion="analytic", ctx=fresh)
        path = str(tmp_path / "r.bbal")
        assert c2b._lib.lib().c2b_write_bal_resident(fresh.handle, path.encode(), 1, None) == INVALID
        assert b"host-buffer" in c2b._lib.lib().c2b_last_error()
        assert not os.path.exists(path)
    finally:
        fresh.close()


# ---- the C++ mirror ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def test_bal_exe(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("cpp") / "test_bal")
    so_dir = os.path.join(ROOT, "city2ba_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_bal.cpp"), "-o", exe, "-L", so_dir,
                           "-lcity2ba_cuda", f"-Wl,-rpath,{so_dir}"])
    return exe


def test_cpp_write_on_gpu_equals_host(test_bal_exe, tmp_path):
    r = subprocess.run([test_bal_exe, str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
