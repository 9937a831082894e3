"""Context lifetime: a context stays usable after a call that failed part-way, several contexts live on different
threads at once, and closing a context and its scene gives its device memory back.

The failing calls are argument and I/O errors that the library reports after it has allocated; nothing here provokes a
device fault or runs the device out of memory."""
import ctypes
import threading

import numpy as np
import pytest

from city2ba_b200.baproblem import IOError_, ParseError
from conftest import bits_equal
from test_gpu_bal import random_problem

pytestmark = pytest.mark.gpu

INVALID = -1


@pytest.fixture
def contexts(c2b):
    """opens explicit Contexts on device 0 (never the process-wide one) and closes them after the test"""
    opened = []

    def open_ctx():
        opened.append(c2b.Context(0))
        return opened[-1]

    yield open_ctx
    for ctx in opened:
        ctx.close()


@pytest.fixture(scope="module")
def cfg2(orc):
    cams, pts = orc.grid_cameras(10, 4), orc.grid_points(10, 4)
    xyz, tri = orc.city_mesh(4)
    return cams, pts, xyz, tri, orc.visibility_graph(xyz, tri, cams, pts, 10.0)


def assert_same_problem(a, b):
    assert (a.num_cameras(), a.num_points(), a.num_observations()) == (b.num_cameras(), b.num_points(),
                                                                       b.num_observations())
    assert bits_equal(a.cameras, b.cameras) and bits_equal(a.points, b.points)
    assert np.array_equal(np.asarray(a.vis_graph.offsets, np.uint64), np.asarray(b.vis_graph.offsets, np.uint64))
    assert np.array_equal(np.asarray(a.vis_graph.point_idx, np.uint64), np.asarray(b.vis_graph.point_idx, np.uint64))
    assert bits_equal(a.vis_graph.uv, b.vis_graph.uv)


def assert_same_graph(a, b):
    assert np.array_equal(np.asarray(a.offsets, np.uint64), np.asarray(b.offsets, np.uint64))
    assert np.array_equal(np.asarray(a.point_idx, np.uint64), np.asarray(b.point_idx, np.uint64))
    assert bits_equal(a.uv, b.uv)


# ---- an error, then a valid call on the same context ---------------------------------------------------------------
def test_cull_after_decreasing_offsets(c2b, contexts):
    rng = np.random.default_rng(51)
    cams, pts = rng.normal(size=(40, 15)), rng.normal(size=(300, 3))
    off = np.arange(0, 41 * 8, 8, dtype=np.uint64)
    off[20] = off[19] - 1  # the CSR offsets decrease
    idx = rng.integers(0, 300, int(off[-1])).astype(np.uint32)
    uv = rng.normal(size=(len(idx), 2))
    ctx = contexts()
    pd = ctypes.POINTER(ctypes.c_double)
    rc = c2b._lib.lib().c2b_cull_problem(ctx.handle, cams.ctypes.data_as(pd), len(cams), pts.ctypes.data_as(pd),
                                         len(pts), off.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)),
                                         idx.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), uv.ctypes.data_as(pd),
                                         ctypes.byref(c2b._lib.CullStats()))
    assert rc == INVALID
    good = random_problem(c2b, rng, 400, 3000, 12)
    assert_same_problem(good.cull_gpu(ctx), good.cull_gpu(contexts()))


def test_read_bal_after_truncated_file(c2b, contexts, tmp_path):
    ba = random_problem(c2b, np.random.default_rng(52), 200, 1500, 10)
    good = str(tmp_path / "good.bal")
    ba.write_text(good)
    data = open(good, "rb").read()
    short = str(tmp_path / "short.bal")
    open(short, "wb").write(data[:len(data) // 2])
    ctx = contexts()
    with pytest.raises(ParseError):
        c2b.BAProblem.from_file_gpu(short, ctx)
    assert_same_problem(c2b.BAProblem.from_file_gpu(good, ctx), c2b.BAProblem.from_file_gpu(good, contexts()))


def test_write_bal_after_missing_directory(c2b, contexts, tmp_path):
    ba = random_problem(c2b, np.random.default_rng(53), 200, 1500, 10)
    ctx = contexts()
    for ext in ("bal", "bbal"):
        with pytest.raises(IOError_):
            ba.write_gpu(str(tmp_path / "missing" / f"x.{ext}"), ctx)
        ba.write_gpu(str(tmp_path / f"a.{ext}"), ctx)
        ba.write_gpu(str(tmp_path / f"b.{ext}"), contexts())
        assert open(tmp_path / f"a.{ext}", "rb").read() == open(tmp_path / f"b.{ext}", "rb").read()


def test_resident_pass_after_unknown_option(c2b, contexts, cfg2):
    cams, pts, xyz, tri, _ = cfg2

    def resident(ctx):
        rp = c2b.generate.ResidentProblem(ctx)
        rp.upload_cameras(cams)
        rp.upload_points(pts)
        return rp, c2b.Scene(xyz, tri, ctx=ctx)

    rp, scene = resident(contexts())
    rp.run(scene, 10.0)
    opt = c2b.generate._options("grid", "mesh", False, False, 20.0, 1.0)
    opt.cull_mode = 7
    assert c2b._lib.lib().c2b_visibility_graph_resident(rp.ctx.handle, scene.handle, 10.0, ctypes.byref(opt),
                                                        ctypes.byref(c2b._lib.Obs())) == INVALID
    rp.run(scene, 10.0)
    rp_ref, scene_ref = resident(contexts())
    rp_ref.run(scene_ref, 10.0)
    assert_same_graph(rp.download(), rp_ref.download())
    scene.close()
    scene_ref.close()


# ---- contexts on several threads ---------------------------------------------------------------------------------
def test_concurrent_contexts(c2b, cfg2):
    cams, pts, xyz, tri, ref = cfg2
    errors = []

    def guarded(fn):
        def run():
            try:
                fn()
            except BaseException as e:  # noqa: BLE001 - reported by the main thread
                errors.append(e)
        return run

    def worker():
        for _ in range(3):
            ctx = c2b.Context(0)
            try:
                scene = c2b.Scene(xyz, tri, ctx=ctx)
                g = c2b.visibility_graph(scene, cams, pts, 10.0, ctx=ctx)
                assert_same_graph(g, ref)
                scene.close()
            finally:
                ctx.close()

    def churn():
        for _ in range(6):
            ctx = c2b.Context(0)
            try:
                c2b.Scene(xyz, tri, ctx=ctx).close()
            finally:
                ctx.close()

    threads = [threading.Thread(target=guarded(f)) for f in (worker, worker, churn)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors


# ---- teardown gives the device memory back ---------------------------------------------------------------------------
def test_teardown_returns_device_memory(c2b, orc):
    import torch
    cams = orc.grid_cameras(10, 4)
    xyz, tri = orc.city_mesh(4)
    grid = orc.grid_points(10, 4)
    lo, hi = grid.min(axis=0) - 1.0, grid.max(axis=0) + 1.0
    P = 16_000_000  # the AoS and SoA copies of the points and the point grid come to about 1.5 GB
    pts = np.random.default_rng(54).uniform(lo, hi, (P, 3))
    free_after = []
    for _ in range(4):
        ctx = c2b.Context(0)
        try:
            scene = c2b.Scene(xyz, tri, ctx=ctx)
            rp = c2b.generate.ResidentProblem(ctx)
            rp.upload_cameras(cams)
            rp.upload_points(pts)
            rp.run(scene, 2.0)
            in_use = torch.cuda.mem_get_info(0)[0]
            scene.close()
        finally:
            ctx.close()
        free_after.append(torch.cuda.mem_get_info(0)[0])
        assert free_after[-1] - in_use > 1 << 30, "the cycle should hold more than 1 GB of device memory"
    assert abs(free_after[-1] - free_after[0]) <= 256 << 20, [f / 2**20 for f in free_after]
