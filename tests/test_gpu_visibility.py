"""Parity tests proper: the CUDA path (through the C ABI) against the CPU oracle and the golden
fixtures.  Bar: bit-exact visibility sets, bit-exact f64 projections (tolerance stated by the
north star is 1e-9 relative; the implementation achieves 0)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, assert_same_graph, points_on_mesh, procedural_scene, random_cameras

pytestmark = pytest.mark.gpu

MODES = ["grid", "exhaustive"]


@pytest.fixture(scope="module")
def cfg2(orc):
    cams, pts = orc.grid_cameras(10, 4), orc.grid_points(10, 4)
    xyz, tri = orc.city_mesh(4)
    return cams, pts, xyz, tri


@pytest.mark.parametrize("mode", MODES)
def test_cfg2_mesh_matches_oracle_and_golden(c2b, ctx, orc, cfg2, mode):
    cams, pts, xyz, tri = cfg2
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    g = c2b.visibility_graph(scene, cams, pts, 10.0, cull_mode=mode, ctx=ctx)
    ref = orc.visibility_graph(xyz, tri, cams, pts, 10.0)
    assert_same_graph(g, ref, f"cfg2/{mode}")
    assert g.stats["n_candidates"] == ref.n_candidates
    gold = np.load(os.path.join(GOLDEN, "cfg2_blocks4.npz"))
    assert np.array_equal(g.offsets, gold["mesh_offsets"]) and np.array_equal(g.point_idx, gold["mesh_idx"])
    assert np.array_equal(g.uv, gold["mesh_uv"])
    if mode == "exhaustive":
        assert g.stats["pairs_evaluated"] == len(cams) * len(pts)
    else:
        assert g.stats["n_candidates"] <= g.stats["pairs_evaluated"] < len(cams) * len(pts)


def test_cfg2_endpoint_guard_and_analytic_and_none(c2b, ctx, orc, cfg2):
    cams, pts, xyz, tri = cfg2
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    gold = np.load(os.path.join(GOLDEN, "cfg2_blocks4.npz"))
    g = c2b.visibility_graph(scene, cams, pts, 10.0, endpoint_guard_rel=True, ctx=ctx)
    assert np.array_equal(g.offsets, gold["guard_offsets"]) and np.array_equal(g.point_idx, gold["guard_idx"])
    a = c2b.visibility_graph(None, cams, pts, 10.0, occlusion="analytic", ctx=ctx)
    assert np.array_equal(a.offsets, gold["analytic_offsets"]) and np.array_equal(a.point_idx, gold["analytic_idx"])
    n = c2b.visibility_graph(None, cams, pts, 10.0, occlusion="none", ctx=ctx)
    assert np.array_equal(n.offsets, gold["cand_offsets"]) and np.array_equal(n.point_idx, gold["cand_idx"])


@pytest.mark.parametrize("mode", MODES)
def test_cfg1_scene_golden(c2b, ctx, mode):
    gold = np.load(os.path.join(GOLDEN, "cfg1_scene.npz"))
    scene = c2b.Scene(gold["xyz"], gold["tri"], ctx=ctx)
    assert scene.num_triangles == len(gold["tri"]) - 2          # two degenerate `l`-style triples dropped
    g = c2b.visibility_graph(scene, gold["cams"], gold["pts"], 100.0, cull_mode=mode, ctx=ctx)
    assert np.array_equal(g.offsets, gold["offsets"]) and np.array_equal(g.point_idx, gold["idx"])
    assert np.array_equal(g.uv, gold["uv"])


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("mode", MODES)
def test_random_scene_matches_oracle(c2b, ctx, orc, seed, mode):
    rng = np.random.default_rng(100 + seed)
    xyz, tri = procedural_scene(seed)
    cams = random_cameras(rng, 50)
    pts = np.concatenate([points_on_mesh(rng, xyz, tri, 700), rng.uniform(-20, 20, (100, 3))])
    md = [15.0, 40.0, 100.0][seed]
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    g = c2b.visibility_graph(scene, cams, pts, md, cull_mode=mode, ctx=ctx)
    ref = orc.visibility_graph(xyz, tri, cams, pts, md)
    assert ref.n_obs > 0 and ref.n_obs < ref.n_candidates
    assert_same_graph(g, ref, f"scene{seed}/{mode}")


def test_triangle_soup_matches_oracle(c2b, ctx, orc):
    """random intersecting triangles: stresses the LBVH (overlapping boxes, duplicate Morton codes)"""
    rng = np.random.default_rng(7)
    xyz = rng.uniform(-10, 10, (400, 3)).astype(np.float32)
    tri = rng.integers(0, 400, (2000, 3)).astype(np.uint32)
    tri[::50] = tri[1::50][: len(tri[::50])]           # exact duplicates -> identical Morton keys
    cams = random_cameras(rng, 64, center=(0, 0, 0), spread=9.0)
    pts = rng.uniform(-10, 10, (1500, 3))
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    for mode in MODES:
        g = c2b.visibility_graph(scene, cams, pts, 30.0, cull_mode=mode, ctx=ctx)
        ref = orc.visibility_graph(xyz, tri, cams, pts, 30.0)
        assert 0 < ref.n_obs < ref.n_candidates
        assert_same_graph(g, ref, f"soup/{mode}")


def test_ray_level_entry_matches_oracle_predicate(c2b, ctx, orc):
    """c2b_occluded (Embree-shaped AoS rays) against a brute-force loop of the oracle predicate"""
    rng = np.random.default_rng(3)
    xyz, tri = procedural_scene(1)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    n = 3000
    org = rng.uniform(-15, 15, (n, 3)).astype(np.float32)
    org[:, 1] = np.abs(org[:, 1]) * 0.2 + 0.1
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d = d.astype(np.float32)
    d[::97, 1] = 0.0                                    # axis-parallel components
    d[5::211] = (1.0, 0.0, 0.0)
    tfar = rng.uniform(0.5, 60, n).astype(np.float32)
    got = scene.occluded(org, d, tfar)
    valid = tri[(tri[:, 0] != tri[:, 1]) & (tri[:, 1] != tri[:, 2]) & (tri[:, 0] != tri[:, 2])]
    want = np.zeros(n, bool)
    for i in range(n):
        ray = np.concatenate([org[i], d[i], tfar[i:i + 1]]).astype(np.float32)
        want[i] = any(orc.ray_triangle(ray, xyz[a], xyz[b], xyz[c]) for a, b, c in valid)
    assert want.any() and not want.all()
    assert np.array_equal(got, want)


def test_intersect1_closest_hit(c2b, ctx):
    xyz = np.array([[-5, 0, -5], [5, 0, -5], [5, 0, 5], [-5, 0, 5], [-5, 2, -5], [5, 2, -5], [5, 2, 5], [-5, 2, 5]], np.float32)
    tri = np.array([[0, 1, 2], [0, 2, 3], [4, 5, 6], [4, 6, 7]], np.uint32)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    hit, t = scene.intersect1([0.5, 10.0, 0.25], [0, -1, 0])
    assert hit and abs(t - 8.0) < 1e-5                  # upper plane first (src/generate.rs:253-262 usage)
    hit, _ = scene.intersect1([50.0, 10.0, 0.0], [0, -1, 0])
    assert not hit
    lo, hi = scene.bounds()
    assert np.array_equal(lo, [-5, 0, -5]) and np.array_equal(hi, [5, 2, 5])


def test_edge_cases(c2b, ctx, orc):
    cams, pts = orc.grid_cameras(2, 1), orc.grid_points(3, 1)
    empty = c2b.Scene(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint32), ctx=ctx)
    assert empty.num_triangles == 0 and empty.num_nodes == 0
    ref = orc.visibility_graph(np.zeros((0, 3)), np.zeros((0, 3)), cams, pts, 10.0)
    for mode in MODES:
        assert_same_graph(c2b.visibility_graph(empty, cams, pts, 10.0, cull_mode=mode, ctx=ctx), ref, "empty scene")
        g = c2b.visibility_graph(empty, cams[:0], pts, 10.0, cull_mode=mode, ctx=ctx)       # no cameras
        assert len(g) == 0 and g.num_observations == 0
        g = c2b.visibility_graph(empty, cams, pts[:0], 10.0, cull_mode=mode, ctx=ctx)       # no points
        assert len(g) == len(cams) and g.num_observations == 0 and np.all(g.offsets == 0)
        g = c2b.visibility_graph(empty, cams, pts, 0.0, cull_mode=mode, ctx=ctx)            # nothing in range
        assert g.num_observations == 0
        g = c2b.visibility_graph(empty, cams, pts, float("inf"), cull_mode=mode, ctx=ctx)   # everything in range
        assert_same_graph(g, orc.visibility_graph(np.zeros((0, 3)), np.zeros((0, 3)), cams, pts, float("inf")), "inf")
    # a single triangle (root is a leaf) and only-degenerate triangles
    one = c2b.Scene(np.array([[5, -1, -30], [5, 5, 0], [5, -1, 30]], np.float32), np.array([[0, 1, 2]], np.uint32), ctx=ctx)
    assert one.num_nodes == 1
    x1 = np.array([[5, -1, -30], [5, 5, 0], [5, -1, 30]], np.float32)
    assert_same_graph(c2b.visibility_graph(one, cams, pts, 30.0, ctx=ctx),
                      orc.visibility_graph(x1, [[0, 1, 2]], cams, pts, 30.0), "one triangle")
    deg = c2b.Scene(x1, np.array([[0, 0, 1], [2, 1, 1]], np.uint32), ctx=ctx)
    assert deg.num_triangles == 0
    # a point sitting exactly on a camera centre, NaN and huge coordinates: same decisions as the oracle
    p2 = np.concatenate([pts, [orc.center(cams[0])], [[np.nan, 0, 0]], [[1e300, 0, 0]]])
    assert_same_graph(c2b.visibility_graph(one, cams, p2, 30.0, ctx=ctx),
                      orc.visibility_graph(x1, [[0, 1, 2]], cams, p2, 30.0), "odd points")
    with pytest.raises(c2b.C2BError):
        c2b.Scene(x1, np.array([[0, 1, 7]], np.uint32), ctx=ctx)                        # vertex out of range
    with pytest.raises(c2b.C2BError):
        c2b.visibility_graph(None, cams, pts, 10.0, occlusion="mesh", ctx=ctx)          # mesh needs a scene


def test_pool_regrows_on_overflow(c2b, orc):
    """a fresh context starts with a small candidate pool; a dense problem must still be exact"""
    ctx2 = c2b.Context(0)
    rng = np.random.default_rng(9)
    cams = random_cameras(rng, 200, spread=2.0)
    pts = rng.uniform(-30, 30, (12000, 3))
    empty = c2b.Scene(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint32), ctx=ctx2)
    g = c2b.visibility_graph(empty, cams, pts, 200.0, cull_mode="exhaustive", ctx=ctx2)
    ref = orc.visibility_graph(np.zeros((0, 3)), np.zeros((0, 3)), cams, pts, 200.0)
    assert ref.n_obs > 300000
    assert_same_graph(g, ref, "overflow")
    ctx2.close()


def test_synthetic_entry_points(c2b, ctx, orc):
    """synthetic_grid / synthetic_line mirrors: same pre-cull graph as the oracle, and the
    reference's own assertion for test_line (tests/main.rs:197-201)"""
    from city2ba_b200 import synthetic
    ba = synthetic.synthetic_grid(10, 20, 3, 5.0, 1.0, 1.0, 1.0, 10.0, False, cull=False, ctx=ctx)
    cams, pts = orc.grid_cameras(10, 3, 5.0, 1.0), orc.grid_points(20, 3, 5.0, 1.0, 1.0)
    ref = orc.synthetic_visibility(cams, pts, 10.0, True, 5.0, 1.0)
    assert_same_graph(ba.vis_graph, ref, "synthetic_grid analytic")
    culled = synthetic.synthetic_grid(10, 20, 3, 5.0, 1.0, 1.0, 1.0, 10.0, False, ctx=ctx)
    assert "Bundle Adjustment Problem" in str(culled) and culled.num_cameras() > 0
    line = synthetic.synthetic_line(30, 40, 10.0, 1.0, 1.0, 1.0, 10.0, False, ctx=ctx)
    assert line.num_cameras() > 20
    lref = orc.synthetic_visibility(orc.line_cameras(30, 10.0, 1.0), orc.line_points(40, 10.0, 1.0, 1.0), 10.0, False)
    lraw = synthetic.synthetic_line(30, 40, 10.0, 1.0, 1.0, 1.0, 10.0, False, cull=False, ctx=ctx)
    assert_same_graph(lraw.vis_graph, lref, "synthetic_line")


@pytest.mark.parametrize("cfg", ["cfg3", "cfg4"])
def test_full_size_properties(c2b, ctx, cfg):
    """BASELINE's full sizes — cfg3: 16x16-block city (9,792 cameras x 998,784 points); cfg4: 64x64
    blocks (99,840 x 9,984,000, the configuration the metric is quoted on) — through size-independent
    properties: grid and exhaustive schedules agree bit for bit, the result is idempotent, indices
    ascend inside each camera, projections lie in the frustum and reproject with zero error, every
    observed pair is within max_dist, and the lattice's translation symmetry shows in the counts."""
    from city2ba_b200 import synthetic
    n, cpb, ppb = {"cfg3": (16, 9, 306), "cfg4": (64, 6, 200)}[cfg]
    cams = synthetic.grid_cameras(cpb, n, 20.0, 1.0)
    pts = synthetic.grid_points(ppb, n, 20.0, 1.0, 1.0)
    scene = c2b.Scene(*synthetic.city_mesh(n), ctx=ctx)
    a = c2b.visibility_graph(scene, cams, pts, 10.0, cull_mode="grid", ctx=ctx)
    b = c2b.visibility_graph(scene, cams, pts, 10.0, cull_mode="exhaustive", ctx=ctx)
    again = c2b.visibility_graph(scene, cams, pts, 10.0, cull_mode="grid", ctx=ctx)
    assert a.num_observations > 1_000_000
    for other in (b, again):
        assert np.array_equal(a.offsets, other.offsets) and np.array_equal(a.point_idx, other.point_idx)
        assert np.array_equal(a.uv, other.uv)
    assert a.stats["n_candidates"] == b.stats["n_candidates"]
    assert b.stats["pairs_evaluated"] == len(cams) * len(pts)
    idx = a.point_idx.astype(np.int64)
    starts = a.offsets[1:-1].astype(np.int64)
    d = np.diff(idx)
    mask = np.ones(len(d), bool)
    mask[starts[(starts > 0) & (starts < len(idx))] - 1] = False
    assert np.all(d[mask] > 0)
    assert np.all(np.abs(a.uv) <= 1.0)
    ba = c2b.BAProblem.from_visibility(cams, pts, a)
    assert ba.total_reprojection_error(1.0) < 1e-6
    # every observed pair is within max_dist of its camera (lattice cameras: centre = -R^T t)
    cam_of = np.repeat(np.arange(len(cams)), np.diff(a.offsets.astype(np.int64)))
    sel = np.random.default_rng(0).choice(len(idx), size=min(len(idx), 2_000_000), replace=False)
    R = cams[cam_of[sel], :9].reshape(-1, 3, 3)              # column-major records: R[k] = column k
    centre = -np.einsum("nij,nj->ni", R, cams[cam_of[sel], 9:12])   # -(R^T t) with R stored transposed
    assert np.all(np.linalg.norm(pts[idx[sel]] - centre, axis=1) < 10.0)
    # translation symmetry of the lattice: an interior column of cameras and the next one (one block
    # further along x) see the same geometry up to coordinate rounding, which only moves the
    # end-point cases (DESIGN.md section 2), so their totals agree closely
    counts = a.counts()
    per_col = 4 * cpb * n + 2 * cpb           # cameras pushed per bx column (src/synthetic.rs:179-210)
    interior = np.arange(3 * per_col, 4 * per_col)
    t0, t1 = counts[interior].sum(), counts[interior + per_col].sum()
    assert counts.max() > 0 and abs(int(t0) - int(t1)) <= 0.05 * t0


@pytest.mark.parametrize("seed", [0, 1])
def test_arbitrary_orientations_and_cell_trimming(c2b, ctx, orc, seed):
    """fully random camera rotations (pitch/roll), anisotropic point clouds, several max_dist:
    the grid schedule's cell-range and front-plane row trimming must never lose a candidate"""
    rng = np.random.default_rng(500 + seed)
    n_c, n_p = 96, 6000
    cams = np.empty((n_c, 15))
    for i in range(n_c):
        v9 = np.concatenate([rng.normal(size=3) * 1.5, [0, 0, 0], [rng.uniform(0.6, 1.6), 0.02, -0.001]])
        cam = orc.from_vec(v9)
        cams[i] = orc.from_position_direction(rng.uniform(-30, 30, 3) * np.array([1, 0.3, 1]), cam[:9])
        cams[i, 12:15] = v9[6:9]
    pts = rng.uniform(-35, 35, (n_p, 3)) * np.array([1, [0.02, 0.5][seed], 1])
    pts[::7, 1] = pts[0, 1]                      # many points on one exact plane
    empty = c2b.Scene(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint32), ctx=ctx)
    for md in (3.0, 11.0, 47.0):
        ref = orc.visibility_graph(np.zeros((0, 3)), np.zeros((0, 3)), cams, pts, md)
        assert ref.n_obs > 0
        for mode in MODES:
            assert_same_graph(c2b.visibility_graph(empty, cams, pts, md, cull_mode=mode, ctx=ctx), ref,
                              f"orient{seed}/{mode}/{md}")


@pytest.mark.parametrize("offset", [0.0, 2.0e4])
def test_image_side_planes_never_lose_a_candidate(c2b, ctx, orc, offset):
    """k1 = k2 = 0 cameras (the BASELINE intrinsics: the plan trims rows by the four side planes of the image
    and by the ball) with fully random rotations and focal lengths that are small, large, negative and zero,
    points placed ON the image border |u| = 1 / |v| = 1 and on the max_dist sphere, near the origin and 20 km
    away from it (the slack of the trimming must scale with the magnitudes): grid schedule = oracle"""
    rng = np.random.default_rng(77)
    focals = [1.0, 0.3, 2.5, -1.2, 0.0, 1.0, 7.0, 1e-3]
    cams = np.empty((64, 15))
    for i in range(len(cams)):
        R = orc.from_vec(np.concatenate([rng.normal(size=3) * 2.0, np.zeros(3), [1.0, 0.0, 0.0]]))[:9]
        cams[i] = orc.from_position_direction(offset + rng.uniform(-12, 12, 3) * np.array([1, 0.4, 1]), R)
        cams[i, 12:15] = (focals[i % len(focals)], 0.0, 0.0)
    pts = [offset + rng.uniform(-25, 25, (5000, 3)) * np.array([1, 0.5, 1])]
    md = 13.0
    for c in cams[:24]:                                   # points constructed on the frustum's faces and the sphere
        f = c[12]
        cen = orc.center(c)
        for _ in range(12):
            z = -rng.uniform(0.5, 12.0)
            s = rng.choice([-1.0, 1.0])
            lim = abs(z / f) if f != 0.0 else 5.0          # |u| = 1  <=>  |x| = |z / f|
            if lim > 25.0:
                continue                                  # (kilometres out for f = 1e-3: would only coarsen the grid)
            x, y = (s * lim, rng.uniform(-1, 1) * lim) if rng.uniform() < 0.5 else (rng.uniform(-1, 1) * lim, s * lim)
            pts.append(orc.to_world(c, np.array([x, y, z]))[None])
            d = rng.normal(size=3)
            pts.append((cen + d / np.linalg.norm(d) * md * rng.choice([1.0, 1.0 - 1e-15, 1.0 + 1e-15]))[None])
    pts = np.concatenate(pts)
    ref = orc.visibility_graph(np.zeros((0, 3)), np.zeros((0, 3)), cams, pts, md)
    assert ref.n_obs > 2000
    empty = c2b.Scene(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint32), ctx=ctx)
    for mode in MODES:
        g = c2b.visibility_graph(empty, cams, pts, md, cull_mode=mode, ctx=ctx)
        assert_same_graph(g, ref, f"side planes/{mode}/{offset}")
    # every candidate was among the evaluated pairs, and the trimming is at work (rows hold a fraction of C x P)
    g = c2b.visibility_graph(empty, cams, pts, md, ctx=ctx)
    assert ref.n_candidates <= g.stats["pairs_evaluated"] < 0.35 * len(cams) * len(pts)


def test_long_segments_use_the_radix_fallback(c2b, ctx, orc):
    """a camera that sees more than 4096 points exceeds the shared-memory segment sort"""
    rng = np.random.default_rng(77)
    cams = random_cameras(rng, 12, spread=1.0)
    pts = rng.uniform(-40, 40, (60000, 3)) * np.array([1, 0.2, 1])
    empty = c2b.Scene(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint32), ctx=ctx)
    g = c2b.visibility_graph(empty, cams, pts, 100.0, cull_mode="grid", ctx=ctx)
    ref = orc.visibility_graph(np.zeros((0, 3)), np.zeros((0, 3)), cams, pts, 100.0)
    assert g.counts().max() > 4096
    assert_same_graph(g, ref, "long segments")


def test_dense_mesh_overflows_triangle_lists(c2b, ctx, orc):
    """more than 128 triangles near a camera: the per-camera lists overflow and the generic
    stackless walk takes over for those cameras"""
    rng = np.random.default_rng(31)
    n = 24
    gx, gz = np.meshgrid(np.linspace(-6, 6, n), np.linspace(-6, 6, n), indexing="ij")
    y = 0.3 * np.sin(gx) * np.cos(gz) + rng.normal(0, 0.02, gx.shape)
    xyz = np.stack([gx, y, gz], axis=-1).reshape(-1, 3).astype(np.float32)
    idx = np.arange(n * n).reshape(n, n)
    a, b, c, d = idx[:-1, :-1].ravel(), idx[1:, :-1].ravel(), idx[1:, 1:].ravel(), idx[:-1, 1:].ravel()
    tri = np.concatenate([np.stack([a, b, c], 1), np.stack([a, c, d], 1)]).astype(np.uint32)
    cams = random_cameras(rng, 40, center=(0, 1.0, 0), spread=5.0)
    pts = points_on_mesh(rng, xyz, tri, 1500) + np.array([0, 0.05, 0])
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    ref = orc.visibility_graph(xyz, tri, cams, pts, 12.0)
    assert 0 < ref.n_obs < ref.n_candidates
    for mode in MODES:
        assert_same_graph(c2b.visibility_graph(scene, cams, pts, 12.0, cull_mode=mode, ctx=ctx), ref, f"dense/{mode}")


def test_list_modes_agree(c2b, ctx, orc, cfg2):
    """the four ways a packet finds its triangles — per-camera records in shared memory (leaf list
    <= 64), per-packet records (<= 128, forced here with the hook hoist_max = 0), the lane = node packet
    traversal of the BVH (list overflow, forced with trilist_cap = 1) and the per-ray stackless
    walk (packet_bvh = 0) — give the same graph"""
    cams, pts, xyz, tri = cfg2
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    ref = orc.visibility_graph(xyz, tri, cams, pts, 10.0)
    assert_same_graph(c2b.visibility_graph(scene, cams, pts, 10.0, ctx=ctx), ref, "hoisted")
    try:
        for form in (0, 1):      # leaf lists built by one thread per camera / one warp per camera (lane = node)
            ctx.tune("trilist_warp", form)
            assert_same_graph(c2b.visibility_graph(scene, cams, pts, 10.0, ctx=ctx), ref, f"trilist form {form}")
        ctx.tune("trilist_warp", -1)
        ctx.tune("hoist_max", 0)
        assert_same_graph(c2b.visibility_graph(scene, cams, pts, 10.0, ctx=ctx), ref, "per-packet records")
        ctx.tune("trilist_cap", 1)
        assert_same_graph(c2b.visibility_graph(scene, cams, pts, 10.0, ctx=ctx), ref, "packet bvh")
        ctx.tune("packet_bvh", 0)
        assert_same_graph(c2b.visibility_graph(scene, cams, pts, 10.0, ctx=ctx), ref, "per-ray walk")
        for name in ("no_such_hook", "epilogue", "fu_occ3"):
            with pytest.raises(c2b.C2BError, match="unknown hook"):
                ctx.tune(name, 1)
    finally:
        ctx.tune("reset", 0)


@pytest.mark.parametrize("parts_log2", ["0", "1", "2"])
def test_camera_tickets_agree(c2b, ctx, orc, cfg2, parts_log2, request):
    """a camera's rows dealt to 1, 2 or 4 tickets (own scratch slice and visible count each, stitched
    back together by the sort/write pass) give the same graph — mesh, analytic and no occlusion, and the
    block-sort / global-sort fallbacks of cameras that see more than 1,024 / 4,096 points"""
    cams, pts, xyz, tri = cfg2
    ctx.tune("parts_log2", int(parts_log2))
    request.addfinalizer(lambda: ctx.tune("reset", 0))
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    assert_same_graph(c2b.visibility_graph(scene, cams, pts, 10.0, ctx=ctx), orc.visibility_graph(xyz, tri, cams, pts, 10.0),
                      f"mesh/{parts_log2}")
    for analytic in (True, False):
        ref = orc.synthetic_visibility(cams, pts, 10.0, analytic)
        g = c2b.visibility_graph(None, cams, pts, 10.0, occlusion="analytic" if analytic else "none", ctx=ctx)
        assert_same_graph(g, ref, f"analytic={analytic}/{parts_log2}")
    # dense points around a few cameras, no occluders: per-camera lists beyond the warp and the block sort
    rng = np.random.default_rng(11)
    few = cams[:6].copy()
    dense = np.array([orc.center(c) for c in few]).repeat(1500, axis=0) + rng.uniform(-6, 6, (9000, 3)) * [1, 0.1, 1]
    ref = orc.synthetic_visibility(few, dense, 10.0, False)
    counts = np.diff(ref.offsets)
    assert counts.max() > 1024
    assert_same_graph(c2b.visibility_graph(None, few, dense, 10.0, occlusion="none", ctx=ctx), ref, f"dense/{parts_log2}")
    # points filling a volume: the max_dist ball covers up to 9 x 9 rows of cells, more than the 32 row ranges
    # the plan stores per camera, so the fused pass recomputes them (the FU_ROWS_MANY path)
    vol = rng.uniform(-14, 14, (20000, 3))
    vcams = random_cameras(rng, 30, center=(0, 0, 0), spread=10.0)
    vcams[:, 10] += rng.uniform(-8, 8, 30)                 # move the cameras in y as well
    ref = orc.synthetic_visibility(vcams, vol, 10.0, False)
    assert ref.n_obs > 1000
    assert_same_graph(c2b.visibility_graph(None, vcams, vol, 10.0, occlusion="none", ctx=ctx), ref, f"volume/{parts_log2}")
    far = np.concatenate([dense, dense + 1e-3, dense - 1e-3, dense + 2e-3])
    ref = orc.synthetic_visibility(few[:2], far, 30.0, False)
    assert np.diff(ref.offsets).max() > 4096
    assert_same_graph(c2b.visibility_graph(None, few[:2], far, 30.0, occlusion="none", ctx=ctx), ref, f"global sort/{parts_log2}")


def test_frustum_edge_classification(c2b, ctx, orc):
    """points constructed to project onto |u| = 1 or |v| = 1 (and a few ulps either side), with and
    without radial distortion: the division-free classification of the cull kernel must fall back
    to the exact operation sequence there and agree with the oracle bit for bit"""
    rng = np.random.default_rng(4242)
    cams = random_cameras(rng, 24, center=(0, 1, 0), spread=3.0)
    cams[:8, 12:15] = (1.0, 0.0, 0.0)            # the BASELINE intrinsics
    cams[8:16, 13:15] = 0.0                       # f != 1, no distortion
    pts = []
    for c in cams:
        R = c[:9].reshape(3, 3).T                 # column-major record -> matrix
        t = c[9:12]
        f = c[12]
        for _ in range(40):
            z = -rng.uniform(0.5, 8.0)
            edge = rng.choice([-1.0, 1.0])
            other = rng.uniform(-1.2, 1.2)
            # undistorted image-plane coordinates that land on the frustum edge when k1 = k2 = 0
            a, b = (edge / f, other / f) if rng.uniform() < 0.5 else (other / f, edge / f)
            pc = np.array([-a * z, -b * z, z])
            p = R.T @ (pc - t)
            for k in (-2, -1, 0, 1, 2):
                pts.append(np.nextafter(p, p + k * np.array([1.0, 1.0, 1.0])) if k else p)
    pts = np.array(pts)
    empty = c2b.Scene(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint32), ctx=ctx)
    ref = orc.visibility_graph(np.zeros((0, 3)), np.zeros((0, 3)), cams, pts, 20.0)
    assert 0 < ref.n_obs < len(cams) * len(pts)
    for mode in MODES:
        assert_same_graph(c2b.visibility_graph(empty, cams, pts, 20.0, cull_mode=mode, ctx=ctx), ref, f"edge/{mode}")


@pytest.mark.parametrize("k", [2, 4, 11])
def test_tessellated_city(c2b, ctx, orc, k):
    """BASELINE config 5 in the small: city blocks whose walls are tessellated k x k and displaced,
    points sampled on the mesh.  k = 2 keeps the per-camera leaf lists short (records hoisted per
    camera), k = 4 lands between 64 and 128 entries for many cameras (per-packet records), k = 11
    overflows the lists (stackless BVH walk).  All must reproduce the brute-force oracle."""
    from city2ba_b200 import synthetic
    import bench
    n = 3
    xyz, tri = synthetic.city_mesh_tessellated(n, k)
    cams = synthetic.grid_cameras(4, n, 20.0, 1.0)
    pts = bench.sample_points_on_walls(xyz, tri, 6000, seed=k)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    ref = orc.visibility_graph(xyz, tri, cams, pts, 10.0)
    assert 0 < ref.n_obs < ref.n_candidates
    for mode in MODES:
        assert_same_graph(c2b.visibility_graph(scene, cams, pts, 10.0, cull_mode=mode, ctx=ctx), ref, f"tess{k}/{mode}")


def test_device_resident_points_entry(c2b, ctx, orc, cfg2):
    """c2b_upload_points_device + c2b_visibility_graph(pts = NULL): the multi-GPU flow where the
    points arrive on the device through an all-gather instead of a host upload"""
    import ctypes as C
    import torch
    from city2ba_b200 import _lib
    from city2ba_b200.generate import _options
    cams, pts, xyz, tri = cfg2
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    ref = orc.visibility_graph(xyz, tri, cams, pts, 10.0)
    L = _lib.lib()
    d_pts = torch.from_numpy(pts).to("cuda:0")
    torch.cuda.synchronize()
    _lib.check(L.c2b_upload_points_device(ctx.handle, d_pts.data_ptr(), len(pts)))
    opt = _options("grid", "mesh", False, False, 20.0, 1.0)
    out = _lib.Obs()
    cam_arr = np.ascontiguousarray(cams)
    _lib.check(L.c2b_visibility_graph(ctx.handle, scene.handle, cam_arr.ctypes.data, len(cams), None, len(pts),
                                      10.0, C.byref(opt), C.byref(out)))
    O = int(out.n_obs)
    assert O == ref.n_obs
    assert np.array_equal(np.ctypeslib.as_array(out.offsets, shape=(len(cams) + 1,)), ref.offsets)
    assert np.array_equal(np.ctypeslib.as_array(out.point_idx, shape=(O,)).astype(np.uint64), ref.point_idx)
    assert np.array_equal(np.ctypeslib.as_array(out.uv, shape=(2 * O,)).reshape(-1, 2), ref.uv)
    # a point count that does not match what is resident is refused
    rc = L.c2b_visibility_graph(ctx.handle, scene.handle, cam_arr.ctypes.data, len(cams), None, len(pts) + 1,
                                10.0, C.byref(opt), C.byref(out))
    assert rc != 0 and b"resident" in L.c2b_last_error()


def test_closest_hit_batch_matches_brute_force(c2b, ctx, orc):
    """c2b_intersect (Embree rtcIntersect1 as a batch, BVH walk) against the brute-force minimum of
    the oracle predicate's t over all triangles; rays that miss stay untouched"""
    rng = np.random.default_rng(9)
    xyz, tri = procedural_scene(3)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    n = 3000
    org = rng.uniform(-20, 20, (n, 3)).astype(np.float32) * np.array([1, 0.2, 1], np.float32) + np.array([0, 3, 0], np.float32)
    d = rng.normal(size=(n, 3))
    d[: n // 3] = [0, -1, 0]                      # the downward placement rays of generate_cameras_poisson
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    hit, t = scene.intersect(org, d)
    # brute force in numpy with the SAME f32 formula as c2b_math.cuh tri_record / ray_tri_record
    valid = tri[(tri[:, 0] != tri[:, 1]) & (tri[:, 1] != tri[:, 2]) & (tri[:, 0] != tri[:, 2])]
    best = np.full(n, np.inf, np.float32)
    f = np.float32
    for a_, b_, c_ in valid:
        A, B, Cc = (xyz[a_] - org).astype(f), (xyz[b_] - org).astype(f), (xyz[c_] - org).astype(f)
        e0, e1, e2 = Cc - A, A - B, B - Cc

        def cross(p, q):
            return np.stack([p[:, 1] * q[:, 2] - p[:, 2] * q[:, 1], p[:, 2] * q[:, 0] - p[:, 0] * q[:, 2],
                             p[:, 0] * q[:, 1] - p[:, 1] * q[:, 0]], 1).astype(f)

        def dot(p, q):  # fmaf chain: exact products accumulated in f64 then rounded once per step
            s0 = (p[:, 0] * q[:, 0]).astype(f)
            s1 = (p[:, 1].astype(np.float64) * q[:, 1].astype(np.float64) + s0.astype(np.float64)).astype(f)
            return (p[:, 2].astype(np.float64) * q[:, 2].astype(np.float64) + s1.astype(np.float64)).astype(f)

        U, V, W = dot(d, cross(e0, Cc + A)), dot(d, cross(e1, A + B)), dot(d, cross(e2, B + Cc))
        T = (f(2.0) * dot(A, cross(e0, e1))).astype(f)
        det = ((U + V).astype(f) + W).astype(f)
        mixed = ((U < 0) | (V < 0) | (W < 0)) & ((U > 0) | (V > 0) | (W > 0))
        Ts = np.where(det < 0, -T, T)
        ok = ~mixed & (det != 0) & (Ts > 0)
        with np.errstate(divide="ignore", invalid="ignore"):
            tt = (Ts / np.abs(det)).astype(f)
        best = np.where(ok & (tt < best), tt, best)
    assert np.array_equal(hit, np.isfinite(best))
    assert hit.sum() > n // 4 and (~hit).sum() > 0
    assert np.array_equal(t[hit], best[hit])


@pytest.mark.parametrize("name", ["cfg1_test_scene.npz", "box_obj.npz"])
@pytest.mark.parametrize("mode", MODES)
def test_reference_meshes_golden(c2b, ctx, name, mode):
    """BASELINE config 1: the reference's own test_scene.obj (100 cameras, 200 points, max_dist 100)
    and tests/box.obj, arrays derived by tests/golden/make_golden_obj.py"""
    from city2ba_b200.generate import generate_world_points_uniform
    g = np.load(os.path.join(GOLDEN, name))
    md = float(g["max_dist"])
    scene = c2b.Scene(g["xyz"], g["tri"], ctx=ctx)           # includes the degenerate `l` triples
    v = c2b.visibility_graph(scene, g["cams"], g["pts"], md, cull_mode=mode, ctx=ctx)
    assert np.array_equal(v.offsets, g["offsets"]) and np.array_equal(v.point_idx, g["idx"])
    assert np.array_equal(v.uv, g["uv"])
    assert v.stats["n_candidates"] == len(g["cand_idx"])
    seed = {"cfg1_test_scene.npz": 20261017, "box_obj.npz": 7}[name]
    assert np.array_equal(generate_world_points_uniform(g["xyz"], g["tri"], g["cams"], len(g["pts"]), md, seed=seed, ctx=ctx), g["pts"])


def test_oversized_batches_are_split(c2b, ctx, orc, cfg2, request):
    """a camera batch whose row points exceed the 32-bit scratch offsets is halved and retried
    (the hook max_pairs lowers the limit so that the path runs at test size); the graph is unchanged"""
    request.addfinalizer(lambda: ctx.tune("reset", 0))
    cams, pts, xyz, tri = cfg2
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    ref = orc.visibility_graph(xyz, tri, cams, pts, 10.0)
    ctx.tune("max_pairs", 20000)                          # 800 cameras x ~90 row points: several splits
    g = c2b.visibility_graph(scene, cams, pts, 10.0, ctx=ctx)
    assert_same_graph(g, ref, "split batches")
    ctx.tune("max_pairs", 10)                             # not even one camera fits: a clean error
    with pytest.raises(c2b.C2BError, match="shard the cameras"):
        c2b.visibility_graph(scene, cams, pts, 10.0, ctx=ctx)


def test_outlier_points_do_not_coarsen_the_grid(c2b, ctx, orc):
    """a handful of far-away vertices (stray geometry of an OBJ scene) used to stretch the point grid's cells
    until the schedule degenerated into ~C x P; the cells now resolve the cameras' reach only and everything
    outside is clamped into the edge cells.  Same graph as the oracle, and a PERFORMANCE assertion: the grid
    schedule evaluates a small fraction of the pairs, about as many as without the outliers."""
    n, cpb, ppb = 8, 5, 40                                   # 1,440 cameras x 34,560 points, 160 m wide
    cams, pts = orc.grid_cameras(cpb, n), orc.grid_points(ppb, n)
    xyz, tri = orc.city_mesh(n)
    far = np.array([[1e7, 3.0, -2e7], [-4e8, 1.0, 5.0], [30.0, 9e6, 40.0], [np.inf, 0.0, 0.0], [12.0, -3e9, 7.0]])
    pts2 = np.concatenate([pts[:1200], far, pts[1200:]])
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    clean = c2b.visibility_graph(scene, cams, pts, 10.0, ctx=ctx)
    g = c2b.visibility_graph(scene, cams, pts2, 10.0, ctx=ctx)
    ref, _ = orc.ref_visibility_graph(xyz, tri, cams, pts2, 10.0)
    assert_same_graph(g, ref, "outliers")
    assert ref.n_obs > 100000 and g.num_observations == clean.num_observations
    assert g.stats["pairs_evaluated"] < 0.05 * len(cams) * len(pts2), g.stats["pairs_evaluated"]
    assert g.stats["pairs_evaluated"] < 1.25 * clean.stats["pairs_evaluated"] + 8 * len(cams)
    # the cached (hinted) grid must not be reused by cameras outside its reach: shift a few cameras far away
    moved = cams.copy()
    for k in range(0, len(moved), 7):
        pos = orc.center(moved[k]) + np.array([1e7 - 40.0, 0.0, -2e7 + 40.0])
        moved[k] = orc.from_position_direction(pos, moved[k][:9])
    g2 = c2b.visibility_graph(scene, moved, pts2, 10.0, ctx=ctx)
    assert_same_graph(g2, orc.ref_visibility_graph(xyz, tri, moved, pts2, 10.0)[0], "outliers, cameras moved")


def mt_reference(orc, xyz, tri, cams, pts, md):
    """the graph under the oracle's Moeller-Trumbore restatement: candidates of the cull that orc_occluded_mt
    (brute force over all triangles) does not call occluded"""
    v = orc.visibility_graph(xyz, tri, cams, pts, md)
    occ = orc.occluded_mt(xyz, tri, cams, pts, v).astype(bool)
    cam_of = np.repeat(np.arange(len(cams)), np.diff(v.cand_offsets.astype(np.int64)))
    keep = ~occ
    off = np.concatenate([[0], np.cumsum(np.bincount(cam_of[keep], minlength=len(cams)))]).astype(np.uint64)
    return off, v.cand_point[keep], v.cand_uv[keep], int(occ.sum()), v


@pytest.mark.parametrize("mode", MODES)
def test_predicate_mt_matches_oracle_mt(c2b, ctx, orc, cfg2, mode):
    """c2b_vis_options::predicate = C2B_PRED_MT (Embree's default intersector, what the reference's scene
    runs): bit for bit the oracle's orc_ray_triangle_mt on the cfg2 lattice, the cfg1-shaped scene, box.obj's
    golden scene and a random scene; the watertight default is unchanged and differs on some rays"""
    cases = [("cfg2", cfg2[2], cfg2[3], cfg2[0], cfg2[1], 10.0)]
    g1 = np.load(os.path.join(GOLDEN, "cfg1_scene.npz"))
    cases.append(("cfg1 scene", g1["xyz"], g1["tri"], g1["cams"], g1["pts"], 100.0))
    gb = np.load(os.path.join(GOLDEN, "box_obj.npz"))
    cases.append(("box.obj", gb["xyz"], gb["tri"], gb["cams"], gb["pts"], float(gb["max_dist"]) if "max_dist" in gb.files else 100.0))
    rng = np.random.default_rng(77)
    xyz, tri = procedural_scene(3)
    cases.append(("random", xyz, tri, random_cameras(rng, 40), points_on_mesh(rng, xyz, tri, 900), 30.0))
    differs = 0
    for name, xyz, tri, cams, pts, md in cases:
        off, idx, uv, n_occ, v = mt_reference(orc, xyz, tri, cams, pts, md)
        scene = c2b.Scene(xyz, tri, ctx=ctx)
        g = c2b.visibility_graph(scene, cams, pts, md, cull_mode=mode, predicate="mt", ctx=ctx)
        assert np.array_equal(g.offsets, off), f"{name}/{mode}: offsets differ under the MT predicate"
        assert np.array_equal(g.point_idx, idx) and np.array_equal(g.uv, uv), f"{name}/{mode}"
        assert g.stats["n_candidates"] == v.n_candidates
        w = c2b.visibility_graph(scene, cams, pts, md, cull_mode=mode, ctx=ctx)
        assert_same_graph(w, v, f"{name}/{mode} watertight default")
        differs += int(w.num_observations != g.num_observations)
    assert differs > 0   # the two predicates do not decide every end-point ray alike (DESIGN.md section 2)


def test_first_call_on_a_fresh_ctx_returns_the_same_graph(c2b, orc, cfg2):
    """the first host-buffer call on a ctx returns its CSR in unpinned memory filled through a pinned ring by host
    threads (pinning a large result costs more than computing it); later calls, and a ctx with the hook
    cold_staged = 0, use pinned arrays — all of them the same graph, with pageable and with large inputs"""
    from city2ba_b200 import _lib
    cams, pts, xyz, tri = cfg2
    ref = orc.visibility_graph(xyz, tri, cams, pts, 10.0)
    for hook in (1, 0):
        fresh = _lib.Context(0)
        try:
            fresh.tune("cold_staged", hook)
            scene = c2b.Scene(xyz, tri, ctx=fresh)
            for call in range(3):
                assert_same_graph(c2b.visibility_graph(scene, cams, pts, 10.0, ctx=fresh), ref, f"cold_staged={hook} call {call}")
            scene.close()
        finally:
            fresh.close()
    # a result large enough for many ring chunks and several camera batches: cfg3 on a fresh ctx, twice
    import bench
    cams3, pts3, xyz3, tri3 = bench.build_workload("cfg3")
    fresh = _lib.Context(0)
    try:
        fresh.tune("batches", 5)
        scene = c2b.Scene(xyz3, tri3, ctx=fresh)
        first = c2b.visibility_graph(scene, cams3, pts3, bench.MAX_DIST, ctx=fresh)
        second = c2b.visibility_graph(scene, cams3, pts3, bench.MAX_DIST, ctx=fresh)
        assert bench.result_hash(first.offsets, first.point_idx, first.uv) == bench.expected_hash("cfg3")
        assert np.array_equal(first.point_idx, second.point_idx) and np.array_equal(first.uv, second.uv)
        scene.close()
    finally:
        fresh.close()
