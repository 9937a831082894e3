"""The point grid's x split (c2b_tune "grid_x_split"): cells 1/k as wide in x as in y and z.  Only the set of points
each camera reads changes, never the result: for every k the whole CSR must be byte-identical to k = 1 — single- and
multi-ticket cameras, cameras with more rows than the plan stores, and a grid whose split the cell budget caps."""
import numpy as np
import pytest

from conftest import assert_same_graph, points_on_mesh, procedural_scene, random_cameras

pytestmark = pytest.mark.gpu

SPLITS = [1, 2, 8, 16]


def graphs_by_split(c2b, ctx, request, run, hooks=()):
    """{k: graph} for every split, with the extra hooks set; the ctx is reset afterwards"""
    request.addfinalizer(lambda: ctx.tune("reset", 0))
    out = {}
    for k in SPLITS:
        ctx.tune("reset", 0)
        for name, value in hooks:
            ctx.tune(name, value)
        ctx.tune("grid_x_split", k)
        out[k] = run()
    return out


def assert_all_identical(gs, what):
    ref = gs[1]
    for k, g in gs.items():
        assert np.asarray(g.offsets).tobytes() == np.asarray(ref.offsets).tobytes(), f"{what}/k={k}: offsets differ"
        assert np.asarray(g.point_idx).tobytes() == np.asarray(ref.point_idx).tobytes(), f"{what}/k={k}: indices differ"
        assert np.asarray(g.uv).tobytes() == np.asarray(ref.uv).tobytes(), f"{what}/k={k}: projections differ"
        assert g.stats["n_candidates"] == ref.stats["n_candidates"], f"{what}/k={k}"


@pytest.fixture(scope="module")
def cfg2(orc):
    cams, pts = orc.grid_cameras(10, 4), orc.grid_points(10, 4)
    xyz, tri = orc.city_mesh(4)
    return cams, pts, xyz, tri


def test_cfg2(c2b, ctx, orc, cfg2, request):
    """800 cameras: fewer than the persistent warps, so each camera's rows are dealt to four tickets"""
    cams, pts, xyz, tri = cfg2
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    gs = graphs_by_split(c2b, ctx, request, lambda: c2b.visibility_graph(scene, cams, pts, 10.0, ctx=ctx))
    assert_same_graph(gs[1], orc.visibility_graph(xyz, tri, cams, pts, 10.0), "cfg2")
    assert_all_identical(gs, "cfg2")


def test_cfg3_and_fewer_pairs(c2b, ctx, request):
    import bench
    cams, pts, xyz, tri = bench.build_workload("cfg3")
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    gs = graphs_by_split(c2b, ctx, request, lambda: c2b.visibility_graph(scene, cams, pts, bench.MAX_DIST, ctx=ctx))
    assert_all_identical(gs, "cfg3")
    p1, p8 = gs[1].stats["pairs_evaluated"], gs[8].stats["pairs_evaluated"]
    assert p8 <= 0.9 * p1, (p1, p8)
    # a shard of a few cameras: one camera's rows over several tickets
    few = cams[:: len(cams) // 300][:300]
    gs = graphs_by_split(c2b, ctx, request, lambda: c2b.visibility_graph(scene, few, pts, bench.MAX_DIST, ctx=ctx))
    assert gs[1].num_observations > 1000
    assert_all_identical(gs, "cfg3 shard")
    scene.close()


@pytest.mark.parametrize("seed", [0, 1])
def test_random_scene(c2b, ctx, orc, seed, request):
    rng = np.random.default_rng(300 + seed)
    xyz, tri = procedural_scene(seed)
    cams = random_cameras(rng, 60)
    pts = np.concatenate([points_on_mesh(rng, xyz, tri, 3000), rng.uniform(-20, 20, (2000, 3))])
    md = [15.0, 40.0][seed]
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    gs = graphs_by_split(c2b, ctx, request, lambda: c2b.visibility_graph(scene, cams, pts, md, ctx=ctx))
    assert_same_graph(gs[1], orc.visibility_graph(xyz, tri, cams, pts, md), f"scene{seed}")
    assert_all_identical(gs, f"scene{seed}")


def test_more_rows_than_the_plan_stores(c2b, ctx, orc, cfg2, request):
    """cells of max_dist / 10: a camera's ball covers up to 21 x 21 rows, more than the 32 row ranges the plan keeps,
    so the fused pass recomputes them 32 at a time"""
    cams, pts, xyz, tri = cfg2
    gs = graphs_by_split(c2b, ctx, request,
                         lambda: c2b.visibility_graph(None, cams, pts, 10.0, occlusion="analytic", ctx=ctx),
                         hooks=[("grid_cell_factor", 0.1)])
    assert_same_graph(gs[1], orc.synthetic_visibility(cams, pts, 10.0, True), "rows")
    assert_all_identical(gs, "rows")
    rng = np.random.default_rng(12)
    vol = rng.uniform(-14, 14, (40000, 3))
    vcams = random_cameras(rng, 30, center=(0, 0, 0), spread=10.0)
    vcams[:, 10] += rng.uniform(-8, 8, 30)
    gs = graphs_by_split(c2b, ctx, request,
                         lambda: c2b.visibility_graph(None, vcams, vol, 10.0, occlusion="none", ctx=ctx),
                         hooks=[("grid_cell_factor", 0.1), ("parts_log2", 0)])
    assert_same_graph(gs[1], orc.synthetic_visibility(vcams, vol, 10.0, False), "volume")
    assert_all_identical(gs, "volume")


def test_split_capped_by_the_cell_budget(c2b, ctx, orc, request):
    """points over 1536 x 32 x 32 m, max_dist 4 (cells 1 m): 1.6 M cells unsplit, 3.1 M at k = 2, 6.3 M at k = 4 —
    over the 2^22 budget, so every k >= 2 builds the k = 2 grid"""
    from oracle import oracle as o
    rng = np.random.default_rng(5)
    pts = rng.uniform(0, 1, (300000, 3)) * [1536.0, 32.0, 32.0]
    cams = np.empty((500, 15))
    for i in range(len(cams)):
        pos = rng.uniform(0, 1, 3) * [1536.0, 24.0, 24.0] + [0.0, 4.0, 4.0]
        R = o.from_axis_angle([0, 1, 0], rng.uniform(0, 2 * np.pi))
        cams[i] = o.from_position_direction(pos, R)
        cams[i, 12:15] = (rng.uniform(0.5, 1.5), 0.0, 0.0)
    gs = graphs_by_split(c2b, ctx, request,
                         lambda: c2b.visibility_graph(None, cams, pts, 4.0, occlusion="none", ctx=ctx))
    assert_same_graph(gs[1], orc.synthetic_visibility(cams, pts, 4.0, False), "capped")
    assert gs[1].num_observations > 1000
    assert_all_identical(gs, "capped")
    pairs = {k: g.stats["pairs_evaluated"] for k, g in gs.items()}
    assert pairs[2] == pairs[8] == pairs[16] < pairs[1], pairs
