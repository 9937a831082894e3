"""Host-side mirror of the reference's library surface (no GPU): lattices, mesh, BAProblem graph
ops, BAL I/O."""
import numpy as np

from conftest import procedural_scene  # noqa: F401


def test_lattices_and_mesh_match_oracle(orc, c2b):
    from city2ba_b200 import synthetic
    for cpb, ppb, n in [(10, 10, 4), (3, 7, 2), (1, 1, 1)]:
        assert np.array_equal(synthetic.grid_cameras(cpb, n, 20.0, 1.0), orc.grid_cameras(cpb, n))
        assert np.array_equal(synthetic.grid_points(ppb, n, 20.0, 1.0, 1.0), orc.grid_points(ppb, n))
        x, t = synthetic.city_mesh(n)
        ox, ot = orc.city_mesh(n)
        assert np.array_equal(x, ox) and np.array_equal(t, ot)
    assert np.array_equal(synthetic.grid_cameras(10, 3, 5.0, 1.0), orc.grid_cameras(10, 3, 5.0, 1.0))
    assert np.array_equal(synthetic.line_cameras(30, 10.0, 1.0), orc.line_cameras(30, 10.0, 1.0))
    assert np.array_equal(synthetic.line_points(40, 10.0, 1.0, 1.0), orc.line_points(40, 10.0, 1.0, 1.0))


def _problem(orc, c2b):
    cams, pts = orc.grid_cameras(10, 3, 5.0, 1.0), orc.grid_points(20, 3, 5.0, 1.0, 1.0)
    v = orc.synthetic_visibility(cams, pts, 10.0, True, 5.0, 1.0)
    g = c2b.VisGraph(v.offsets, v.point_idx, v.uv)
    return c2b.BAProblem.from_visibility(cams, pts, g)


def test_baproblem_cull_invariants(orc, c2b):
    ba = _problem(orc, c2b)
    culled = ba.cull()
    g = culled.vis_graph
    assert culled.num_cameras() <= ba.num_cameras() and culled.num_points() <= ba.num_points()
    assert np.all(g.counts() > 3)                      # cameras see >= 4 points (src/baproblem.rs:432)
    pc = np.bincount(g.point_idx.astype(np.int64), minlength=culled.num_points())
    assert np.all(pc > 1)                              # points seen at least twice (:448)
    again = culled.cull()                              # fixed point (:542)
    assert again.num_cameras() == culled.num_cameras() and again.num_points() == culled.num_points()
    assert culled.total_reprojection_error(2.0) < 1e-12
    assert str(culled).startswith("Bundle Adjustment Problem with ")


def test_baproblem_list_of_lists_round_trip(orc, c2b):
    ba = _problem(orc, c2b)
    lol = [ba.vis_graph[i] for i in range(5)] + [[] for _ in range(ba.num_cameras() - 5)]
    ba2 = c2b.BAProblem.from_visibility(ba.cameras, ba.points, lol)
    assert ba2.vis_graph[3] == ba.vis_graph[3]
    assert ba2.num_observations() == sum(len(x) for x in lol)


def test_bal_binary_and_text_round_trip(orc, c2b, tmp_path):
    ba = _problem(orc, c2b).cull()
    for ext in ("bbal", "bal"):
        path = tmp_path / f"p.{ext}"
        ba.write(path)
        back = c2b.BAProblem.from_file(path)
        assert back.num_cameras() == ba.num_cameras() and back.num_points() == ba.num_points()
        assert np.array_equal(back.vis_graph.offsets, ba.vis_graph.offsets)
        assert np.array_equal(back.vis_graph.point_idx, ba.vis_graph.point_idx)
        assert np.array_equal(back.vis_graph.uv, ba.vis_graph.uv)      # shortest round-trip text
        assert np.array_equal(back.points, ba.points)
        assert np.allclose(back.cameras, ba.cameras, atol=1e-12)        # through Rodrigues vectors
    head = open(tmp_path / "p.bal").readline().split()
    assert [int(x) for x in head] == [ba.num_cameras(), ba.num_points(), ba.num_observations()]
    raw = open(tmp_path / "p.bbal", "rb").read()
    assert int.from_bytes(raw[:8], "big") == ba.num_cameras()           # big-endian (src/baproblem.rs:738)


def test_text_format_never_uses_exponent(c2b, tmp_path):
    cams = np.zeros((1, 15))
    cams[0, [0, 4, 8, 12]] = 1.0
    g = c2b.VisGraph(np.array([0, 1], np.uint64), np.array([0], np.uint64), np.array([[1e-7, 0.30000000000000004]]))
    ba = c2b.BAProblem(cams, np.array([[1e21, -2.5e-9, 1.0]]), g)
    ba.write(tmp_path / "x.bal")
    txt = open(tmp_path / "x.bal").read()
    assert "e" not in txt.lower() and "0.0000001" in txt and "0.30000000000000004" in txt


def _write_obj(path):
    """quads, a pentagon, relative indices, v/vt/vn forms and a poly-line object (the shape of the reference's
    tests/box.obj); the same text tests/cpp/test_host.cpp writes"""
    lines = ["# test scene", "mtllib none.mtl", "o Plane", "v -4 0 -4", "v 4 0 -4", "v 4 0 4", "v -4 0 4", "vn 0 1 0",
             "usemtl None", "s off", "f 1//1 2//1 3//1 4//1", "o Cube"]
    for k in range(8):
        lines.append(f"v {1 if k & 1 else -1} {2 if k & 2 else 0} {1 if k & 4 else -1}")
    lines += ["f 5 6 8 7", "f 9 11 12 10", "f 5 9 10 6", "f 7 8 12 11", "f 5 7 11 9", "f -7 -5 -1 -3",
              "o Roof", "v -1 2 -1", "v 1 2 -1", "v 1.5 2 0", "v 1 2 1", "v -1 2 1", "f 13 14 15 16 17", "o Curve"]
    lines += [f"v {-3.0 + k} 0.5 3" for k in range(6)] + [f"l {18 + k} {19 + k}" for k in range(5)]
    open(path, "w").write("\n".join(lines) + "\n")


def _dump(models):
    out = []
    for m in models:
        p = m.positions.reshape(-1).astype(np.float64)
        ps = float((p * (1 + np.arange(len(p)) % 7)).sum())
        s = int((m.indices.astype(np.uint64) * (1 + np.arange(len(m.indices), dtype=np.uint64) % 5)).sum())
        out.append((m.name, len(m.positions), len(m.indices), ps, s))
    return out


def _write_golden_mesh_obj(path, name):
    """the reference's own meshes (test_scene.obj, tests/box.obj) as tests/golden stores them, after tobj's
    triangulation, written back as OBJ text: one object, one `f` record per stored index triple (the triples
    the `l` records left are degenerate ones); returns the stored (xyz, tri)"""
    import os
    from conftest import GOLDEN
    g = np.load(os.path.join(GOLDEN, name))
    lines = ["o Mesh"] + ["v %r %r %r" % tuple(float(x) for x in v) for v in g["xyz"]]
    lines += ["f %d %d %d" % tuple(int(k) + 1 for k in t) for t in g["tri"]]
    open(path, "w").write("\n".join(lines) + "\n")
    return g["xyz"], g["tri"]


def test_obj_loader_python_equals_cpp(c2b, tmp_path):
    """the two host mirrors read OBJ files identically (tobj 0.1.12's rules): the hand-written scene and the
    reference's own meshes from tests/golden, which both must read back to the stored triangles"""
    import os
    import subprocess
    from conftest import ROOT
    from city2ba_b200 import generate
    exe = str(tmp_path / "test_host")
    so_dir = os.path.join(ROOT, "city2ba_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_host.cpp"), "-o", exe, "-L", so_dir,
                           "-lcity2ba_cuda", f"-Wl,-rpath,{so_dir}"])
    mine = str(tmp_path / "scene.obj")
    _write_obj(mine)
    files = [mine]
    for name in ("box_obj.npz", "cfg1_test_scene.npz"):
        f = str(tmp_path / name.replace(".npz", ".obj"))
        xyz, tri = _write_golden_mesh_obj(f, name)
        lx, lt = generate.concat_models(generate.load_obj(f))
        assert np.array_equal(lx[lt], xyz[tri]), name     # the same triangles, corner for corner
        files.append(f)
    for f in files:
        cpp = []
        for line in subprocess.check_output([exe, "obj", f], text=True).splitlines():
            name, nv, ni, ps, s = line.split("|")
            cpp.append((name, int(nv), int(ni), float(ps), int(s)))
        py = _dump(generate.load_obj(f))
        assert [(a[0], a[1], a[2], a[4]) for a in py] == [(a[0], a[1], a[2], a[4]) for a in cpp], f
        assert np.allclose([a[3] for a in py], [a[3] for a in cpp], rtol=1e-8), f
    models = generate.load_obj(mine)
    assert [m.name for m in models] == ["Plane", "Cube", "Roof", "Curve"]
    assert list(models[2].indices) == [0, 1, 2, 0, 2, 3, 0, 3, 4]               # fan
    assert list(models[3].indices) == [0, 1, 1, 2, 2, 3, 3, 4, 4, 5]            # `l` records: index pairs
    xyz, tri = generate.concat_models(models)
    assert xyz.shape == (23, 3) and tri.shape == (20, 3)
    assert generate.move_to_origin(models)[1].positions.min() >= 0.0
    import pytest
    with pytest.raises(c2b.baproblem.IOError_):
        generate.load_obj(str(tmp_path / "missing.obj"))


def test_graph_noise_python_mirror(c2b, orc):
    """src/noise.rs:180-378 through the Python mirror: the reference's library properties (tests/main.rs:155-190)
    on a problem whose projections are exact"""
    from city2ba_b200 import noise
    ba = _problem(orc, c2b).cull()
    e0 = ba.total_reprojection_error(2.0)
    n_obs = ba.vis_graph.num_observations
    mis = noise.add_incorrect_correspondences(ba, 0.01, seed=4)
    assert mis.vis_graph.num_observations == n_obs and mis.total_reprojection_error(2.0) > e0
    assert np.array_equal(np.sort(mis.vis_graph.point_idx), np.sort(ba.vis_graph.point_idx))
    dropped = noise.drop_features(ba, 0.1, seed=5)
    assert np.array_equal(dropped.vis_graph.counts(), (ba.vis_graph.counts() * 0.1).astype(np.int64))
    assert dropped.total_reprojection_error(2.0) >= e0 - 1e-9
    split = noise.split_landmarks(ba, 0.1, seed=6)
    assert split.num_points() == ba.num_points() + int(0.1 * ba.num_points())
    assert split.total_reprojection_error(2.0) >= e0 - 1e-9 and abs(split.total_reprojection_error(2.0) - e0) < 1e-9
    assert (split.vis_graph.point_idx >= ba.num_points()).sum() > 0
    joined = noise.join_landmarks(ba, 0.01, seed=7)
    changed = joined.vis_graph.point_idx != ba.vis_graph.point_idx
    assert 0 < changed.sum() <= int(0.01 * ba.num_points()) and joined.total_reprojection_error(2.0) > e0
