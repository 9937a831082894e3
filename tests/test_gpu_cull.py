"""BAProblem::cull on the GPU (c2b_cull_problem / c2b_cull_problem_resident) against the host mirror
BAProblem.cull(): identical camera records, points, CSR and (u, v) bits, and the same number of applications of
largest_connected_component + remove_singletons."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, bits_equal, points_on_mesh, procedural_scene, random_cameras

pytestmark = pytest.mark.gpu

INVALID = -1


# ---- helpers -------------------------------------------------------------------------------------------------
def host_cull(ba):
    """BAProblem.cull() with the loop of src/baproblem.rs:538-549 spelled out, counting the applications"""
    nc, npt = ba.num_cameras(), ba.num_points()
    culled, it = ba.largest_connected_component().remove_singletons(), 1
    while (culled.num_cameras(), culled.num_points()) != (nc, npt):
        nc, npt = culled.num_cameras(), culled.num_points()
        culled, it = culled.largest_connected_component().remove_singletons(), it + 1
    return culled, it


def quirk_drops(ba):
    """per application of the loop: does the :523 filter (label of the point index, no camera offset) drop an
    observation of a camera of the largest component?"""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    out, cur, prev = [], ba, None
    while prev is None or (cur.num_cameras(), cur.num_points()) != prev:
        prev = (cur.num_cameras(), cur.num_points())
        nc, npt = prev
        if nc:
            g = cur.vis_graph
            cam_of = np.repeat(np.arange(nc), g.counts())
            idx = g.point_idx.astype(np.int64)
            A = coo_matrix((np.ones(len(idx), np.int8), (cam_of, idx + nc)), shape=(nc + npt, nc + npt))
            _, lab = connected_components(A, directed=False)
            L = int(np.argmax(np.bincount(lab)))
            out.append(bool(np.any((lab[cam_of] == L) & (lab[idx] != L))))
        else:
            out.append(False)
        cur = cur.largest_connected_component().remove_singletons()
    return out


def assert_same_problem(a, b, what=""):
    assert (a.num_cameras(), a.num_points(), a.num_observations()) == \
        (b.num_cameras(), b.num_points(), b.num_observations()), what
    assert bits_equal(a.cameras, b.cameras), f"{what}: camera records differ"
    assert bits_equal(a.points, b.points), f"{what}: points differ"
    assert np.array_equal(np.asarray(a.vis_graph.offsets, np.uint64), np.asarray(b.vis_graph.offsets, np.uint64)), \
        f"{what}: offsets differ"
    assert np.array_equal(np.asarray(a.vis_graph.point_idx, np.uint64), np.asarray(b.vis_graph.point_idx, np.uint64)), \
        f"{what}: point indices differ"
    assert bits_equal(a.vis_graph.uv, b.vis_graph.uv), f"{what}: (u, v) differ"


def check_gpu_equals_host(c2b, ctx, ba, what=""):
    ref, it = host_cull(ba)
    st = {}
    got = ba.cull_gpu(ctx, stats=st)
    assert_same_problem(got, ref, what)
    assert st["iterations"] == it, f"{what}: {st['iterations']} applications on the GPU, {it} on the host"
    return ref, it


def make_problem(c2b, rng, per_camera, P):
    """per_camera: list of point-index lists; cameras and points with random (distinct) bits"""
    C = len(per_camera)
    cams = rng.normal(size=(C, 15))
    pts = rng.normal(size=(P, 3))
    off = np.zeros(C + 1, np.uint64)
    off[1:] = np.cumsum([len(o) for o in per_camera])
    idx = np.array([p for o in per_camera for p in o], np.uint64)
    uv = rng.normal(size=(len(idx), 2))
    uv[rng.random(len(idx)) < 0.1] *= -0.0  # signed zeros travel as bits
    return c2b.BAProblem(cams, pts, c2b.VisGraph(off, idx, uv))


def random_problem(c2b, rng):
    """several components (groups of cameras over disjoint point sets), equal-sized groups now and then,
    duplicates, unsorted lists, cameras with 0-5+ observations, isolated points"""
    n_groups = int(rng.integers(1, 5))
    P = int(rng.integers(0, 60))
    perm = rng.permutation(P)
    cuts = np.sort(rng.integers(0, P + 1, n_groups - 1)) if P else np.zeros(n_groups - 1, int)
    groups = np.split(perm[: max(P - int(rng.integers(0, 4)), 0)], cuts) if P else [np.zeros(0, int)] * n_groups
    per_camera = []
    for _ in range(int(rng.integers(0, 40))):
        gp = groups[int(rng.integers(0, len(groups)))]
        k = int(rng.integers(0, 9)) if len(gp) else 0
        per_camera.append([int(x) for x in rng.choice(gp, size=k, replace=True)] if k else [])
    return make_problem(c2b, rng, per_camera, P)


def tie_problem(c2b, rng):
    """two (or three) components of exactly the same size, interleaved in the numbering"""
    k = int(rng.integers(2, 4))
    nc, npg = int(rng.integers(2, 6)), int(rng.integers(2, 8))
    per_camera = []
    for c in range(nc * k):
        g = c % k
        pts = [g + k * j for j in range(npg)]  # group g owns points g, g + k, ...
        per_camera.append([int(p) for p in rng.permutation(pts)])
    return make_problem(c2b, rng, per_camera, npg * k)


def peeling_chain(c2b, rng, n):
    """camera 0 has 3 observations; camera i shares point s_{i-1} with camera i-1 and s_i with camera i+1 and sees
    its own point q_i twice (duplicates count): every application peels one camera or one point off the chain"""
    s = list(range(n))                 # shared points s_0 .. s_{n-1}
    q = list(range(n, 2 * n + 1))      # private points q_0 .. q_n
    r = 2 * n + 1
    per_camera = [[s[0], q[0], q[0]]]
    for i in range(1, n):
        per_camera.append([s[i - 1], q[i], s[i], q[i]])
    per_camera.append([s[n - 1], q[n], q[n], r, r])
    return make_problem(c2b, rng, per_camera, 2 * n + 2)


def late_quirk(c2b, rng):
    """cluster A (cameras first in the numbering) and cluster B (points first) joined by a camera with 3
    observations: the first application keeps everything but that camera; in the second, B is the larger
    component and its observations of points 0..5 — entities 0..5 are A's cameras — fall to the :523 filter"""
    a_cams, b_cams, a_pts, b_pts = 6, 10, 5, 8
    A = [b_pts + j for j in range(a_pts)]
    B = list(range(b_pts))
    per_camera = [list(rng.permutation(A)) for _ in range(a_cams)]
    per_camera.append([A[0], B[0], B[1]])
    per_camera += [list(rng.permutation(B)) for _ in range(b_cams)]
    return make_problem(c2b, rng, per_camera, a_pts + b_pts)


# ---- 1-3: hand-made, random and edge-case graphs ----------------------------------------------------------------
def test_hand_made_quirk_graph(c2b, ctx):
    """the problem of test_cpp_host.py::test_python_mirror_lcc_matches_reference_quirk"""
    cams = np.zeros((3, 15))
    cams[:, [0, 4, 8, 12]] = 1.0
    pts = np.array([[0.5 * i, 0.1 * i, -3.0 - 0.2 * i] for i in range(6)])
    idx = np.tile(np.arange(5, dtype=np.uint64), 2)
    ba = c2b.BAProblem(cams, pts, c2b.VisGraph(np.array([0, 5, 10, 10], np.uint64), idx, np.zeros((10, 2))))
    ref, _ = check_gpu_equals_host(c2b, ctx, ba, "hand-made")
    assert (ref.num_cameras(), ref.num_points(), ref.num_observations()) == (2, 4, 8)


def test_random_graphs(c2b, ctx):
    rng = np.random.default_rng(2024)
    quirk, multi = 0, 0
    for t in range(300):
        ba = random_problem(c2b, rng)
        _, it = check_gpu_equals_host(c2b, ctx, ba, f"random graph {t}")
        quirk += any(quirk_drops(ba))
        multi += it > 1
    assert quirk > 10 and multi > 10, (quirk, multi)  # the cases the test is meant to cover did occur


def test_large_random_graphs(c2b, ctx):
    """tens of thousands of entities in a few long-range components: deep union-find trees and many threads
    resolving the same roots at once in the label pass"""
    rng = np.random.default_rng(31)
    for t in range(6):
        C, P, groups = 40000, 20000, int(rng.integers(1, 4))
        grp_of_pt = rng.integers(0, groups, P)
        by_grp = [np.nonzero(grp_of_pt == g)[0] for g in range(groups)]
        k = rng.integers(0, 12, C)
        g_of_cam = rng.integers(0, groups, C)
        per_camera = [[int(x) for x in rng.choice(by_grp[g], size=int(n))] for g, n in zip(g_of_cam, k)]
        check_gpu_equals_host(c2b, ctx, make_problem(c2b, rng, per_camera, P), f"large graph {t}")


def test_equal_components_lowest_label_wins(c2b, ctx):
    rng = np.random.default_rng(7)
    for t in range(40):
        ba = tie_problem(c2b, rng)
        check_gpu_equals_host(c2b, ctx, ba, f"tie {t}")
        lcc = ba.largest_connected_component()  # the first application's choice: camera 0's component
        assert lcc.num_cameras() == ba.num_cameras() // (ba.num_points() // lcc.num_points())
        assert bits_equal(lcc.cameras[0], ba.cameras[0])


def test_peeling_chain(c2b, ctx):
    rng = np.random.default_rng(3)
    for n in (2, 3, 5, 9):
        _, it = check_gpu_equals_host(c2b, ctx, peeling_chain(c2b, rng, n), f"chain {n}")
        assert it >= 3


def test_quirk_after_renumbering(c2b, ctx):
    ba = late_quirk(c2b, np.random.default_rng(5))
    drops = quirk_drops(ba)
    assert not drops[0] and any(drops[1:]), drops
    check_gpu_equals_host(c2b, ctx, ba, "late quirk")


@pytest.mark.parametrize("case", ["no_cameras", "no_points", "no_observations", "few_observations"])
def test_edge_cases(c2b, ctx, case):
    rng = np.random.default_rng(11)
    if case == "no_cameras":
        ba = make_problem(c2b, rng, [], 5)
    elif case == "no_points":
        ba = make_problem(c2b, rng, [[], [], []], 0)
    elif case == "no_observations":
        ba = make_problem(c2b, rng, [[], [], []], 4)
    else:
        ba = make_problem(c2b, rng, [[int(p) for p in rng.integers(0, 6, int(rng.integers(0, 4)))] for _ in range(12)], 6)
    check_gpu_equals_host(c2b, ctx, ba, case)
    c0 = make_problem(c2b, rng, [], 0)
    check_gpu_equals_host(c2b, ctx, c0, "empty")


# ---- 4-5: real graphs through the resident chain ------------------------------------------------------------------
def _cfg2_inputs(c2b):
    from city2ba_b200 import synthetic
    cams = synthetic.grid_cameras(10, 4, 20.0, 1.0)
    pts = synthetic.grid_points(10, 4, 20.0, 1.0, 1.0)
    return cams, pts


def _resident(c2b, ctx, cams, pts, scene, **kw):
    rp = c2b.generate.ResidentProblem(ctx)
    rp.upload_cameras(cams)
    rp.upload_points(pts)
    rp.run(scene, 10.0, **kw)
    return rp


def _resident_cull_equals_host(c2b, ctx, cams, pts, scene, what, **kw):
    rp = _resident(c2b, ctx, cams, pts, scene, **kw)
    g = rp.download()
    ba = c2b.BAProblem(cams, pts, g)
    ref, it = host_cull(ba)
    st = rp.cull()
    assert st["iterations"] == it, what
    assert (st["n_cameras"], st["n_points"], st["n_obs"]) == (ref.num_cameras(), ref.num_points(), ref.num_observations())
    c, p = rp.download_problem(st["n_cameras"], st["n_points"])
    got = c2b.BAProblem(c, p, rp.download())
    assert_same_problem(got, ref, what)
    return rp, ref


def test_resident_cfg2(c2b, ctx):
    from city2ba_b200 import synthetic
    cams, pts = _cfg2_inputs(c2b)
    _resident_cull_equals_host(c2b, ctx, cams, pts, None, "cfg2 analytic", occlusion="analytic")
    xyz, tri = synthetic.city_mesh(4)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    _resident_cull_equals_host(c2b, ctx, cams, pts, scene, "cfg2 mesh")


def test_resident_procedural_scene(c2b, ctx):
    rng = np.random.default_rng(1)
    xyz, tri = procedural_scene(0)
    cams = random_cameras(rng, 300)
    pts = points_on_mesh(rng, xyz, tri, 3000)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    _resident_cull_equals_host(c2b, ctx, cams, pts, scene, "procedural")


def test_resident_cfg3_full_size(c2b, ctx):
    from city2ba_b200 import synthetic
    cams = synthetic.grid_cameras(9, 16, 20.0, 1.0)
    pts = synthetic.grid_points(306, 16, 20.0, 1.0, 1.0)
    xyz, tri = synthetic.city_mesh(16)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    _resident_cull_equals_host(c2b, ctx, cams, pts, scene, "cfg3")


def test_state_after_resident_cull(c2b, ctx):
    rng = np.random.default_rng(4)
    xyz, tri = procedural_scene(0)
    cams = random_cameras(rng, 300)
    pts = points_on_mesh(rng, xyz, tri, 3000)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    rp, ref = _resident_cull_equals_host(c2b, ctx, cams, pts, scene, "state")
    assert ref.num_observations() > 0
    # reprojection error of the culled problem
    assert rp.reprojection_error(2.0) == pytest.approx(ref.total_reprojection_error(2.0), rel=1e-12, abs=1e-15)
    # culling again: a fixed point
    st = rp.cull()
    assert st["iterations"] == 1
    assert (st["n_cameras"], st["n_points"], st["n_obs"]) == (ref.num_cameras(), ref.num_points(), ref.num_observations())
    c, p = rp.download_problem(ref.num_cameras(), ref.num_points())
    assert_same_problem(c2b.BAProblem(c, p, rp.download()), ref, "second cull")
    # a second resident pass equals a fresh ctx's pass on the culled cameras and points
    rp.run(scene, 10.0)
    again = rp.download()
    fresh = c2b.Context(0)
    try:
        s2 = c2b.Scene(xyz, tri, ctx=fresh)
        rp2 = _resident(c2b, fresh, ref.cameras, ref.points, s2)
        g2 = rp2.download()
        assert np.array_equal(again.offsets, g2.offsets) and np.array_equal(again.point_idx, g2.point_idx)
        assert bits_equal(again.uv, g2.uv)
        s2.close()
    finally:
        fresh.close()
    # resident add_noise after the cull equals the host-buffer pass on the downloaded culled problem
    rp = _resident(c2b, ctx, cams, pts, scene)
    rp.cull()
    rp.add_noise(0.01, 0.001, 0.01, 0.001, seed=9)
    c, p = rp.download_problem(ref.num_cameras(), ref.num_points())
    g = rp.download()
    hc, hp, huv = ref.cameras.copy(), ref.points.copy(), ref.vis_graph.uv.copy()
    pd = ctypes.POINTER(ctypes.c_double)
    L = c2b._lib.lib()
    c2b._lib.check(L.c2b_add_noise(ctx.handle, hc.ctypes.data_as(pd), len(hc), hp.ctypes.data_as(pd), len(hp),
                                   huv.ctypes.data_as(pd), len(huv), 0.01, 0.001, 0.01, 0.001, 9))
    assert bits_equal(c, hc) and bits_equal(p, hp) and bits_equal(g.uv, huv)


def test_host_entry_leaves_resident_problem_alone(c2b, ctx):
    cams, pts = _cfg2_inputs(c2b)
    rp = _resident(c2b, ctx, cams, pts, None, occlusion="analytic")
    before = rp.download()
    cb, pb = rp.download_problem(len(cams), len(pts))
    rng = np.random.default_rng(12)
    for _ in range(3):
        check_gpu_equals_host(c2b, ctx, random_problem(c2b, rng), "beside a resident problem")
    after = rp.download()
    ca, pa = rp.download_problem(len(cams), len(pts))
    assert np.array_equal(before.offsets, after.offsets) and np.array_equal(before.point_idx, after.point_idx)
    assert bits_equal(before.uv, after.uv) and bits_equal(cb, ca) and bits_equal(pb, pa)


# ---- 7: errors ------------------------------------------------------------------------------------------------
def _raw_cull(c2b, ctx, cams, pts, off, idx, uv):
    pd = ctypes.POINTER(ctypes.c_double)
    st = c2b._lib.CullStats()
    return c2b._lib.lib().c2b_cull_problem(ctx.handle, cams.ctypes.data_as(pd), len(cams), pts.ctypes.data_as(pd),
                                            len(pts), off.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)),
                                            idx.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)),
                                            uv.ctypes.data_as(pd), ctypes.byref(st))


@pytest.mark.parametrize("bad", ["first_offset", "decreasing", "index_range"])
def test_invalid_input_is_rejected_untouched(c2b, ctx, bad):
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
    copies = [a.copy() for a in (cams, pts, off, idx, uv)]
    assert _raw_cull(c2b, ctx, cams, pts, off, idx, uv) == INVALID
    for a, b in zip((cams, pts, off, idx, uv), copies):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


def test_resident_cull_without_result(c2b):
    fresh = c2b.Context(0)
    try:
        st = c2b._lib.CullStats()
        assert c2b._lib.lib().c2b_cull_problem_resident(fresh.handle, ctypes.byref(st)) == INVALID
        cams, pts = _cfg2_inputs(c2b)
        rp = c2b.generate.ResidentProblem(fresh)
        rp.upload_cameras(cams)
        rp.upload_points(pts)
        assert c2b._lib.lib().c2b_cull_problem_resident(fresh.handle, ctypes.byref(st)) == INVALID
    finally:
        fresh.close()


def test_resident_cull_after_host_buffer_call(c2b):
    fresh = c2b.Context(0)
    try:
        cams, pts = _cfg2_inputs(c2b)
        c2b.visibility_graph(None, cams, pts, 10.0, occlusion="analytic", ctx=fresh)
        st = c2b._lib.CullStats()
        assert c2b._lib.lib().c2b_cull_problem_resident(fresh.handle, ctypes.byref(st)) == INVALID
        assert b"host-buffer" in c2b._lib.lib().c2b_last_error()
    finally:
        fresh.close()


# ---- 8: the C++ mirror ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def test_cull_exe(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("cpp") / "test_cull")
    so_dir = os.path.join(ROOT, "city2ba_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_cull.cpp"), "-o", exe, "-L", so_dir,
                           "-lcity2ba_cuda", f"-Wl,-rpath,{so_dir}"])
    return exe


def test_cpp_cull_on_gpu_equals_host(test_cull_exe):
    r = subprocess.run([test_cull_exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "test_cull ok" in r.stdout
