"""bench.py's checking helpers on the CPU: the result hash must be additive over camera ranges (so that it is the
same however the cameras were split over GPUs) and sensitive to any change of the CSR; parity_against must report
exactly the cameras whose rows differ from the oracle's."""
import numpy as np

import bench
from conftest import bits_equal


def _graph(orc):
    cams, pts = orc.grid_cameras(10, 4), orc.grid_points(10, 4)
    xyz, tri = orc.city_mesh(4)
    return cams, pts, xyz, tri, orc.visibility_graph(xyz, tri, cams, pts, 10.0)


def test_result_hash_is_additive_and_sensitive(orc):
    _, _, _, _, v = _graph(orc)
    h = bench.result_hash(v.offsets, v.point_idx, v.uv)
    off = v.offsets.astype(np.int64)
    for cuts in ([333], [100, 101, 640], [1, 2, 3, 799]):
        total, lo = 0, 0
        for hi in cuts + [len(off) - 1]:
            total += bench.result_hash(off[lo:hi + 1] - off[lo], v.point_idx[off[lo]:off[hi]], v.uv[off[lo]:off[hi]], cam0=lo, chunk=97)
            lo = hi
        assert total & (2 ** 64 - 1) == h
    uv = v.uv.copy()
    uv[5, 0] = np.nextafter(uv[5, 0], 2.0)
    assert bench.result_hash(v.offsets, v.point_idx, uv) != h                  # one ulp in one projection
    idx = v.point_idx.copy()
    idx[[0, 1]] = idx[[1, 0]]
    assert bench.result_hash(v.offsets, idx, v.uv) != h                          # order inside a camera
    off2 = v.offsets.copy()
    k = int(np.nonzero(np.diff(off) > 1)[0][0])
    off2[k + 1] -= 1                                                             # an observation moved to the next camera
    assert bench.result_hash(off2, v.point_idx, v.uv) != h
    assert bench.result_hash(np.zeros(4, np.uint64), np.zeros(0, np.uint32), np.zeros((0, 2))) == \
        bench.result_hash(np.zeros(4, np.uint64), np.zeros(0, np.uint32), np.zeros((0, 2)), chunk=2)


def test_parity_against_counts_differing_cameras(orc):
    cams, pts, xyz, tri, v = _graph(orc)
    sample = np.unique(np.linspace(0, len(cams) - 1, 50).astype(np.int64))
    ref, _ = orc.ref_visibility_graph(xyz, tri, cams[sample], pts, 10.0)
    ok = bench.parity_against(sample, ref, v.offsets, v.point_idx, v.uv)
    assert ok["mismatches"] == 0 and ok["cameras_checked"] == len(sample) and ok["observations_checked"] == ref.n_obs
    uv = v.uv.copy()
    row = int(v.offsets[sample[7]])
    uv[row, 1] += 1e-12
    assert bench.parity_against(sample, ref, v.offsets, v.point_idx, uv)["mismatches"] == 1
    # the sign of a zero counts: the synthetic city has v = +0 for the observations at camera height
    uv = v.uv.copy()
    off = v.offsets.astype(np.int64)
    rows = np.concatenate([np.arange(off[c], off[c + 1]) for c in sample])
    zero = rows[uv[rows, 1] == 0.0]
    assert len(zero) > 0
    uv[zero[0], 1] = -0.0
    assert np.array_equal(uv, v.uv)  # invisible to a value comparison
    assert bench.parity_against(sample, ref, v.offsets, v.point_idx, uv)["mismatches"] == 1
    # what the bench hands over: the flat (2 * O,) view of the library's uv array
    assert bench.parity_against(sample, ref, v.offsets, v.point_idx, v.uv.reshape(-1))["mismatches"] == 0


def test_dump_outputs_whole_and_sampled(orc, tmp_path, monkeypatch):
    _, _, _, _, v = _graph(orc)
    bench.dump_outputs(tmp_path / "all", v.offsets, v.point_idx, v.uv.reshape(-1))
    load = lambda d, n: np.load(tmp_path / d / f"{n}.npy")  # noqa: E731
    assert all(load("all", n).dtype == np.float64 for n in ("offsets", "point_idx", "uv"))
    assert np.array_equal(load("all", "offsets"), v.offsets) and np.array_equal(load("all", "point_idx"), v.point_idx)
    assert bits_equal(load("all", "uv"), v.uv) and load("all", "uv").shape == v.uv.shape
    monkeypatch.setattr(bench, "DUMP_MAX_OBS", 1000)
    for d in ("s1", "s2"):
        bench.dump_outputs(tmp_path / d, v.offsets, v.point_idx, v.uv)
    assert np.array_equal(load("s1", "point_idx"), load("s2", "point_idx"))   # the same seeded sample
    n = len(load("s1", "point_idx"))
    assert 900 < n <= 1000 and load("s1", "uv").shape == (n, 2)
    assert np.isin(load("s1", "point_idx"), v.point_idx.astype(np.float64)).all()


def test_native_oracle_builds_outside_the_checkout():
    """the bench's CPU arm builds the oracle -march=native where it runs; the checkout may be read-only"""
    import os
    import subprocess
    import sys
    from conftest import ROOT
    here = os.path.join(ROOT, "oracle")
    before = sorted(os.listdir(here))
    subprocess.check_call([sys.executable, "-c", "from oracle import oracle as o; assert o.lib().orc_deg_to_rad(180.0) > 3"],
                          cwd=ROOT, env={**os.environ, "C2B_ORACLE_NATIVE": "1", "PYTHONDONTWRITEBYTECODE": "1"})
    assert sorted(os.listdir(here)) == before


def test_workload_generators_agree():
    """the product's host generators and the oracle's build the same lattices (the reference arm uses the latter)"""
    a = bench.build_workload("cfg2", gen="product")
    b = bench.build_workload("cfg2", gen="oracle")
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_bits_equal_sees_what_array_equal_does_not():
    from conftest import bits_equal
    a = np.array([[0.0, 1.5], [np.nan, -2.0]])
    assert bits_equal(a, a.copy()) and not np.array_equal(a, a.copy())  # a NaN equals itself bit for bit
    b = a.copy()
    b[0, 0] = -0.0
    assert np.array_equal(a[0], b[0]) and not bits_equal(a, b)
    assert not bits_equal(a, a[:1])
