"""Noise pass on the GPU against the oracle's identical Philox stream.  Points and observations: BIT-EXACT
(the draws are table + polynomial evaluations with every operation explicit on both sides).  Cameras: 1e-9
relative (sin / cos / pow of libm inside from_axis_angle / from_angle_x differ by a few ulp between glibc and
CUDA's libm)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, assert_same_graph

pytestmark = pytest.mark.gpu
RTOL, ATOL = 1e-9, 1e-12


@pytest.fixture(scope="module")
def problem(c2b, orc):
    cams, pts = orc.grid_cameras(10, 4), orc.grid_points(10, 4)
    gold = np.load(os.path.join(GOLDEN, "cfg2_blocks4.npz"))
    g = c2b.VisGraph(gold["mesh_offsets"], gold["mesh_idx"].astype(np.uint64), gold["mesh_uv"])
    return c2b.BAProblem.from_visibility(cams, pts, g)


def test_mean_std(problem, orc, ctx):
    m, s = problem.mean_std(ctx)
    assert np.allclose(m, orc.mean(problem.cameras, problem.points), rtol=1e-12)
    assert np.allclose(s, orc.std(problem.cameras, problem.points), rtol=1e-12)


def test_drift_deterministic_case_matches_oracle_and_golden(c2b, problem, orc, ctx):
    # cfg2: --drift-strength 0.001, drift std 0 => Normal(1,0) == 1: fully deterministic
    out = c2b.noise.add_drift_normalized(problem, 0.001, 0.0, 0.0, seed=1, ctx=ctx)
    oc, op = orc.add_drift_normalized(problem.cameras, problem.points, 0.001, 0.0, 0.0, 1)
    assert np.allclose(out.cameras, oc, rtol=RTOL, atol=ATOL) and np.allclose(out.points, op, rtol=RTOL, atol=ATOL)
    gold = np.load(os.path.join(GOLDEN, "cfg2_noise.npz"))
    assert np.allclose(out.cameras, gold["drift_cams"], rtol=RTOL, atol=ATOL)
    assert np.allclose(out.points, gold["drift_pts"], rtol=RTOL, atol=ATOL)


def test_drift_random_case(c2b, problem, orc, ctx):
    out = c2b.noise.add_drift(problem, 0.002, 0.0005, 0.3, [0.0, 1.0, 0.5], seed=99, ctx=ctx)
    oc, op = orc.add_drift(problem.cameras, problem.points, 0.002, 0.0005, 0.3, [0.0, 1.0, 0.5], 99)
    assert np.allclose(out.cameras, oc, rtol=RTOL, atol=ATOL) and np.array_equal(out.points, op)
    assert not np.allclose(out.points, problem.points)


def test_add_noise_matches_oracle_and_golden(c2b, problem, orc, ctx):
    out = c2b.noise.add_noise(problem, 0.01, 0.0001, 0.01, 0.001, seed=42, ctx=ctx)
    oc, op, ouv = orc.add_noise(problem.cameras, problem.points, problem.vis_graph.uv, 0.01, 0.0001, 0.01, 0.001, 42)
    assert np.allclose(out.cameras, oc, rtol=RTOL, atol=ATOL)
    assert np.array_equal(out.points, op)                 # bit-exact
    assert np.array_equal(out.vis_graph.uv, ouv)          # bit-exact
    gold = np.load(os.path.join(GOLDEN, "cfg2_noise.npz"))
    assert np.allclose(out.cameras, gold["noise_cams"], rtol=RTOL, atol=ATOL)
    assert np.array_equal(out.points, gold["noise_pts"]) and np.array_equal(out.vis_graph.uv, gold["noise_uv"])


def test_add_noise_streams_observations_in_chunks(c2b, orc, ctx):
    """5 M observations cross the GPU in several chunks (upload, kernel and download of neighbouring chunks
    overlap); element i must still draw from counter i: bit-exact against the oracle"""
    n = 5_000_000
    cams = np.zeros((2, 15))
    cams[:, [0, 4, 8, 12]] = 1.0
    pts = np.arange(9.0).reshape(3, 3)
    uv = np.linspace(-1, 1, 2 * n).reshape(n, 2)
    g = c2b.VisGraph(np.array([0, n // 2, n], np.uint64), np.zeros(n, np.uint64), uv)
    out = c2b.noise.add_noise(c2b.BAProblem(cams, pts, g), 0.0, 0.0, 0.0, 0.01, seed=9, ctx=ctx)
    _, _, ouv = orc.add_noise(cams, pts, uv, 0.0, 0.0, 0.0, 0.01, 9)
    assert np.array_equal(out.vis_graph.uv, ouv)
    assert np.array_equal(out.points, pts)                # point_std 0: untouched


def test_resident_noise_equals_host_entries(c2b, orc, ctx):
    """generate -> noise without leaving HBM (c2b_add_*_resident): the same numbers as the host-array entries"""
    from city2ba_b200.generate import ResidentProblem
    cams, pts = orc.grid_cameras(10, 4), orc.grid_points(10, 4)
    xyz, tri = orc.city_mesh(4)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    rp = ResidentProblem(ctx)
    rp.upload_points(pts)
    rp.upload_cameras(cams)
    rp.run(scene, 10.0)
    g0 = rp.download()
    e0 = rp.reprojection_error(2.0)
    assert e0 < 1e-9
    rp.add_drift(0.001, 0.0, 0.0, None, seed=46)
    rp.add_noise(0.01, 0.0001, 0.01, 0.001, seed=47)
    rc, rpts = rp.download_problem(len(cams), len(pts))
    g1 = rp.download()
    oc, op = orc.add_drift_normalized(cams, pts, 0.001, 0.0, 0.0, 46)
    oc, op, ouv = orc.add_noise(oc, op, g0.uv, 0.01, 0.0001, 0.01, 0.001, 47)
    assert np.allclose(rc, oc, rtol=RTOL, atol=ATOL)
    assert np.allclose(rpts, op, rtol=1e-12, atol=1e-15)      # the drifted cameras' few-ulp differences reach bal.std()
    assert np.array_equal(g1.uv, ouv) and np.array_equal(g1.point_idx, g0.point_idx)
    # the resident reprojection error now measures the noised problem (src/baproblem.rs:265-279)
    # exact sum of the terms of the downloaded problem, within the device reduction's rounding bound
    from city2ba_b200.baproblem import _project_all
    from test_gpu_noise_reductions import reproj_tolerance
    d = np.abs(_project_all(rc, rpts, g0.offsets, g0.point_idx) - g1.uv)
    want, tol, _ = reproj_tolerance((d * d).sum(axis=1), 2.0)
    e1 = rp.reprojection_error(2.0)
    assert e1 > e0 and abs(e1 - want) <= tol
    # and a second visibility pass runs on the noised problem (grid rebuilt, centres refreshed)
    rp.run(scene, 10.0)
    assert_same_graph(rp.download(), orc.visibility_graph(xyz, tri, rc, rpts, 10.0), "after resident noise")


def test_noise_is_distributionally_gaussian(c2b, ctx):
    # 2e5 points, sigma 0.5: displacement magnitude |N(0, sigma)|, direction uniform on the sphere
    n = 200_000
    cams = np.zeros((1, 15))
    cams[0, [0, 4, 8, 12]] = 1.0
    g = c2b.VisGraph(np.array([0, n], np.uint64), np.arange(n, dtype=np.uint64), np.zeros((n, 2)))
    ba = c2b.BAProblem(cams, np.zeros((n, 3)), g)
    out = c2b.noise.add_noise(ba, 0.0, 0.0, 0.5, 0.25, seed=5, ctx=ctx)
    d = out.points
    r = np.linalg.norm(d, axis=1)
    assert abs(r.mean() - 0.5 * np.sqrt(2 / np.pi)) < 5e-3 and abs(np.sqrt((r ** 2).mean()) - 0.5) < 5e-3
    assert np.all(np.abs((d / r[:, None]).mean(axis=0)) < 1e-2)
    ro = np.linalg.norm(out.vis_graph.uv, axis=1)
    assert abs(np.sqrt((ro ** 2).mean()) - 0.25) < 3e-3
    # different seeds differ, same seed repeats
    again = c2b.noise.add_noise(ba, 0.0, 0.0, 0.5, 0.25, seed=5, ctx=ctx)
    other = c2b.noise.add_noise(ba, 0.0, 0.0, 0.5, 0.25, seed=6, ctx=ctx)
    assert np.array_equal(again.points, out.points) and not np.array_equal(other.points, out.points)


def test_reference_library_properties(c2b, ctx):
    """tests/main.rs:130-150: drift and noise must increase the total reprojection error"""
    from city2ba_b200 import synthetic
    ba = synthetic.synthetic_grid(10, 20, 3, 5.0, 1.0, 1.0, 1.0, 10.0, False, ctx=ctx)
    e0 = ba.total_reprojection_error(2.0)
    assert c2b.noise.add_drift_normalized(ba, 0.1, 0.1, 0.1, seed=3, ctx=ctx).total_reprojection_error(2.0) > e0
    assert c2b.noise.add_noise(ba, 0.1, 0.1, 0.1, 0.1, seed=3, ctx=ctx).total_reprojection_error(2.0) > e0


def test_sin_noise_matches_oracle(c2b, problem, orc, ctx):
    # the two calls of run_noise (src/bin/city2ba.rs:319-332): dir x then z, displacement along +y
    for d in ([1.0, 0.0, 0.0], [0.0, 0.0, 1.0], [0.3, -0.2, 0.9]):
        out = c2b.noise.add_sin_noise(problem, d, [0.0, 2.0, 0.0], 0.05, 1.5, ctx=ctx)
        oc, op = orc.add_sin_noise(problem.cameras, problem.points, d, [0.0, 2.0, 0.0], 0.05, 1.5)
        assert np.allclose(out.cameras, oc, rtol=RTOL, atol=ATOL) and np.allclose(out.points, op, rtol=RTOL, atol=ATOL)
        assert not np.allclose(out.points, problem.points)
        assert np.array_equal(out.points[:, [0, 2]], problem.points[:, [0, 2]])  # +y only
    up, kern, down = c2b.noise.last_timing(ctx)
    assert up >= 0 and kern > 0 and down >= 0


def test_sin_noise_flat_dimension_and_property(c2b, ctx):
    """a problem with zero extent in y divides by 1e-8 there (src/noise.rs:395-396), and
    tests/main.rs:185-195: sin noise must increase the total reprojection error"""
    from city2ba_b200 import synthetic
    ba = synthetic.synthetic_grid(10, 20, 3, 5.0, 1.0, 1.0, 1.0, 10.0, False, ctx=ctx)
    e0 = ba.total_reprojection_error(2.0)
    assert c2b.noise.add_sin_noise(ba, [1.0, 0.0, 0.0], [0.0, 1.0, 0.0], 0.1, 1.0, ctx=ctx).total_reprojection_error(2.0) > e0
    cams = np.zeros((2, 15))
    cams[:, [0, 4, 8, 12]] = 1.0
    cams[1, 9] = -3.0                              # centre (3, 0, 0)
    pts = np.array([[1.0, 0.0, 2.0], [2.0, 0.0, -1.0]])
    g = c2b.VisGraph(np.array([0, 0, 0], np.uint64), np.zeros(0, np.uint64), np.zeros((0, 2)))
    out = c2b.noise.add_sin_noise(c2b.BAProblem(cams, pts, g), [0.0, 1.0, 0.0], [1.0, 0.0, 0.0], 0.5, 1.0, ctx=ctx)
    assert np.allclose(out.points, pts)            # y = 0 everywhere: sin(0) = 0
