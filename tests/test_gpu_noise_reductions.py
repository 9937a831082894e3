"""The noise pass's device reductions and resident entries against exact references, at sizes where every
stage of the reductions runs: several grid-stride iterations per thread, full and partial blocks, the one-warp
fold of all 592 block partials.

Statistic references are exact sums (math.fsum) of terms built with the same IEEE operation the kernel applies
to each term (e / num, (e - mean)^2, |u - u'|^p), so only the summation order differs from the GPU.

Tolerance.  The reductions (c2b_noise.cuh) run 592 x 256 = 151,552 threads.  A sum of n terms passes through
  - the per-thread grid-stride loop: ceil(n / 151,552) additions,
  - the warp shuffle tree: 5,
  - the sequential fold of the 8 warp sums of a block: 8,
  - the one-warp strided fold of the 592 block partials: ceil(592 / 32) = 19,
  - the final shuffle tree: 5,
so every term meets at most k = ceil(n / 151,552) + 37 roundings of relative size 2^-53, and
    |gpu - fsum| <= (k + 3) * 2^-53 * sum(|terms|).
The resident reprojection error adds the host's sequential fold of up to 592 partials (k + 592).  The +3 covers
nvcc's default FMA contraction in device code (the build passes -ffp-contract=off to the host compiler only),
which changes a term's rounding by at most one ulp, and a few ulp of CUDA's pow against glibc's.

Every check also asserts that its tolerance is below the change that dropping or doubling one element of its
input would make, so a reduction that loses or repeats an element fails."""
import math

import numpy as np
import pytest

from conftest import assert_same_graph, bits_equal

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
THREADS = 592 * 256                       # ST_BLOCKS x ST_THREADS of the statistic kernels
RTOL, ATOL = 1e-9, 1e-12                  # cameras (libm sin / cos / pow inside), as in test_gpu_noise.py


def fsum(x) -> float:
    return math.fsum(memoryview(np.ascontiguousarray(x, np.float64).reshape(-1)))


def rel_bound(n: int, host_fold: int = 0) -> float:
    """relative bound (k + 3) 2^-53 of a device sum of n terms (see the module docstring)"""
    k = -(-n // THREADS) + 5 + 8 + -(-592 // 32) + 5 + host_fold
    return (k + 3) * U


def reproj_tolerance(terms, norm: float):
    """(exact reference, tolerance) of c2b_reprojection_error_resident, whose result is pow(S, 1/norm) with S the
    device sum of the per-observation terms |du|^p + |dv|^p.  A relative error e of S moves S^(1/p) by e / p; glibc's
    pow on the host rounds the reference and the result the same way up to an ulp each.  Also returns the sum's
    own absolute tolerance, for the sensitivity checks."""
    terms = np.asarray(terms, np.float64)
    s = fsum(terms)
    e = rel_bound(terms.size, host_fold=592)
    ref = s ** (1.0 / norm)
    return ref, (e / norm + 4 * U) * ref, e * s


# ---- problems with known centres ------------------------------------------------------------------------------
def cams_at(centres):
    """identity-rotation cameras: centre = -t exactly (checked against orc.center on a sample)"""
    centres = np.asarray(centres, np.float64).reshape(-1, 3)
    c = np.zeros((len(centres), 15))
    c[:, [0, 4, 8, 12]] = 1.0
    c[:, 9:12] = -centres
    return c


def check_centres(orc, cams, centres):
    for i in np.unique(np.linspace(0, len(cams) - 1, 7).astype(np.int64)) if len(cams) else []:
        assert bits_equal(orc.center(cams[i]), centres[i])


def mean_std(c2b, ctx, chain, C):
    from city2ba_b200.baproblem import BAProblem
    cams = cams_at(chain[:C])
    return BAProblem(cams, np.ascontiguousarray(chain[C:]), None).mean_std(ctx), cams


CFG3_N, CFG4_N = 1_008_576, 10_083_840
SIZES = [1, 2, 31, 32, 33, 255, 256, 257, THREADS - 1, THREADS, THREADS + 1, 2 * THREADS + 7, CFG3_N, CFG4_N]


def splits(n):
    """C = 0, P = 0 (while the cameras stay small enough to hold), and C just before / after a block boundary"""
    out = {0}
    if n <= 2 * THREADS + 7:
        out.add(n)
    out.update(c for c in (255, 257) if c < n and (c == 257 or n <= CFG3_N))
    if n <= 257:
        out.add(n // 2)
    return sorted(out)


def chain_data(family, n, seed):
    rng = np.random.default_rng(seed)
    sign = rng.choice([-1.0, 1.0], size=(n, 3))
    if family == "offset":
        # a large common offset with a small spread; no element within 0.25 of the offset, so no (e - mean)^2 is
        # near zero and every element moves both sums by far more than the tolerance
        return 1e6 + sign * rng.uniform(0.25, 1.0, (n, 3))
    if family == "mixed":
        return sign * 10.0 ** rng.uniform(0.0, 3.0, (n, 3))
    raise ValueError(family)


def check_mean_std(c2b, ctx, chain, C):
    n = len(chain)
    (m, sd), cams = mean_std(c2b, ctx, chain, C)
    num = float(n)
    e = rel_bound(n)
    for a in range(3):
        t = chain[:, a] / num                                    # the kernel's e.x / num, term for term
        assert abs(m[a] - fsum(t)) <= e * fsum(np.abs(t)), (a, m[a], fsum(t))
        assert e * fsum(np.abs(t)) < np.abs(t).min()             # a dropped / doubled element is seen
        d = chain[:, a] - m[a]                                   # the kernel's (e - mean)^2 with the device mean
        q = d * d
        s = fsum(q)
        want = math.sqrt(s / num)
        if n == 1:
            assert sd[a] == 0.0
            continue
        assert abs(sd[a] - want) <= (e / 2 + 4 * U) * want, (a, sd[a], want)
        assert e * s < q.min()
    # the fold order is fixed: a second call gives the same bits
    (m2, sd2), _ = mean_std(c2b, ctx, chain, C)
    assert bits_equal(m, m2) and bits_equal(sd, sd2)
    return cams


@pytest.mark.parametrize("family", ["offset", "mixed"])
@pytest.mark.parametrize("n", SIZES)
def test_mean_std_exact(c2b, orc, ctx, n, family):
    chain = chain_data(family, n, seed=n)
    for C in splits(n):
        cams = check_mean_std(c2b, ctx, chain, C)
        check_centres(orc, cams, chain[:C])


def boundary_positions(n, C):
    """0, C - 1, C, n - 1 and k * 151,552 +- 1 inside [0, n)"""
    pos = {0, C - 1, C, n - 1}
    for k in range(1, n // THREADS + 1):
        pos.update((k * THREADS - 1, k * THREADS + 1))
    return sorted(p for p in pos if 0 <= p < n)


@pytest.mark.parametrize("n,C", [(2 * THREADS + 7, 257), (CFG3_N, 9_792)])
def test_mean_std_sentinel(c2b, ctx, n, C):
    """one element 1e4 among +-[1, 2]: losing it at any boundary position moves the mean and std far"""
    rng = np.random.default_rng(7)
    base = rng.choice([-1.0, 1.0], size=(n, 3)) * rng.uniform(1.0, 2.0, (n, 3))
    for p in boundary_positions(n, C):
        chain = base.copy()
        chain[p] = 1e4
        check_mean_std(c2b, ctx, chain, C)


# ---- the drift origin: nearest element to the world origin, the later index on a tie -------------------------
DRIFT_N, DRIFT_C = 2 * THREADS + 7, 257
DRIFT_DIR = [0.3, -0.5, 0.8]


def far_chain(n, seed):
    """elements 10 to 20 from the origin, in random directions (no two at the same distance)"""
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n, 3))
    return d / np.linalg.norm(d, axis=1)[:, None] * rng.uniform(10.0, 20.0, n)[:, None]


def host_drift(c2b, ctx, chain, C, std, angle, seed=5):
    from city2ba_b200.baproblem import BAProblem
    out = c2b.noise.add_drift(BAProblem(cams_at(chain[:C]), chain[C:], None), 1e-3, angle, std, DRIFT_DIR,
                              seed=seed, ctx=ctx)
    return out.cameras, out.points


def resident_drift(ctx, chain, C, std, angle, direction=DRIFT_DIR, seed=5):
    from city2ba_b200.generate import ResidentProblem
    rp = ResidentProblem(ctx)
    rp.upload_points(chain[C:])
    rp.upload_cameras(cams_at(chain[:C]))
    rp.add_drift(1e-3, angle, std, direction, seed=seed)
    return rp.download_problem(C, len(chain) - C)


def check_drift_origin(c2b, orc, ctx, chain, C, other):
    """`other` is the chain with its nearest element moved away, as a reduction that lost it would see it"""
    cams = cams_at(chain[:C])
    oc, op = orc.add_drift(cams, chain[C:], 1e-3, 0.0, 0.0, DRIFT_DIR, 5)
    _, op_other = orc.add_drift(cams_at(other[:C]), other[C:], 1e-3, 0.0, 0.0, DRIFT_DIR, 5)
    keep = np.all(chain[C:] == other[C:], axis=1)
    assert not bits_equal(op[keep], op_other[keep])              # the origin shows in the points it did not move
    hc, hp = host_drift(c2b, ctx, chain, C, 0.0, 0.0)
    assert bits_equal(hp, op)
    assert np.allclose(hc, oc, rtol=RTOL, atol=ATOL)
    # resident, explicit direction, random magnitudes: the same bits as the host entry
    hc, hp = host_drift(c2b, ctx, chain, C, 0.3, 0.2)
    rc, rpts = resident_drift(ctx, chain, C, 0.3, 0.2)
    assert bits_equal(rc, hc) and bits_equal(rpts, hp)


@pytest.mark.parametrize("pos", sorted(set(boundary_positions(DRIFT_N, DRIFT_C)) | {31, 32, 255}))
def test_drift_origin_unique(c2b, orc, ctx, pos):
    chain = far_chain(DRIFT_N, seed=pos)
    chain[pos] = [0.6, -0.48, 0.64]                              # |.| = 1
    other = chain.copy()
    other[pos] *= 30.0                                           # a reduction that skipped pos: the next nearest
    check_drift_origin(c2b, orc, ctx, chain, DRIFT_C, other)


TIES = {
    "lanes": (3, 17), "warps": (5, 200), "blocks": (10, 1000), "strides": (100, THREADS + 100),
    "seam": (DRIFT_C - 1, DRIFT_C), "cam_pt": (5, DRIFT_C + 5), "ends": (0, DRIFT_N - 1),
    "last_stride": (THREADS - 1, 2 * THREADS + 6),
}


@pytest.mark.parametrize("where", list(TIES))
def test_drift_origin_tie_later_wins(c2b, orc, ctx, where):
    """(a, b, c) and (-a, b, c) have bitwise-equal magnitudes: the later index is the origin (DESIGN.md section 6)"""
    i, j = TIES[where]
    chain = far_chain(DRIFT_N, seed=len(where))
    chain[i] = [-0.6, -0.48, 0.64]
    chain[j] = [0.6, -0.48, 0.64]
    assert np.linalg.norm(chain[i]) == np.linalg.norm(chain[j])
    other = chain.copy()
    other[j] = [6.0, -4.8, 6.4]                                  # without the tie the earlier element is the origin
    check_drift_origin(c2b, orc, ctx, chain, DRIFT_C, other)


# ---- extent (add_sin_noise) -------------------------------------------------------------------------------------
SIN = ([0.6, -0.7, 0.4], [0.2, 1.0, -0.3], 0.05, 1.5)
N = DRIFT_N
EXTENT_CASES = {
    # name: (low, high of the bulk, {axis: (position of the min, position of the max)}, constant axes)
    "boundaries": (-5.0, 5.0, {0: (0, N - 1), 1: (DRIFT_C - 1, DRIFT_C), 2: (THREADS - 1, THREADS + 1)}, {}),
    "strides": (-5.0, 5.0, {0: (2 * THREADS - 1, 2 * THREADS + 1), 1: (31, 32), 2: (255, 256)}, {}),
    "negative": (-30.0, -20.0, {0: (N - 1, 0), 1: (DRIFT_C, DRIFT_C - 1), 2: (THREADS + 1, THREADS - 1)}, {}),
    "one_flat": (-5.0, 5.0, {0: (DRIFT_C - 1, N - 1), 1: (0, THREADS + 1)}, {2: -1.25}),
    "two_flat": (-5.0, 5.0, {0: (DRIFT_C, THREADS - 1)}, {1: 2.5, 2: -1.25}),
}


def extent_chain(name):
    lo, hi, ext, flat = EXTENT_CASES[name]
    rng = np.random.default_rng(len(name))
    chain = rng.uniform(lo, hi, (N, 3))
    for a, (pmin, pmax) in ext.items():
        chain[pmin, a] = lo - 3.0
        chain[pmax, a] = hi + 4.0
    for a, v in flat.items():
        chain[:, a] = v
    return chain


@pytest.mark.parametrize("name", list(EXTENT_CASES))
def test_sin_noise_extent(c2b, orc, ctx, name):
    from city2ba_b200.baproblem import BAProblem
    from city2ba_b200.generate import ResidentProblem
    chain, C = extent_chain(name), DRIFT_C
    cams, pts = cams_at(chain[:C]), chain[C:]
    oc, op = orc.add_sin_noise(cams, pts, *SIN)
    # an extent off by one element moves every result past the tolerance
    _, _, ext, _ = EXTENT_CASES[name]
    for a, ps in ext.items():
        for p in ps:
            moved = chain.copy()
            moved[p, a] = 0.5 * (EXTENT_CASES[name][0] + EXTENT_CASES[name][1])
            _, mp = orc.add_sin_noise(cams_at(moved[:C]), moved[C:], *SIN)
            keep = np.arange(C, N) != p
            assert not np.allclose(mp[keep], op[keep], rtol=RTOL, atol=ATOL), (a, p)
    out = c2b.noise.add_sin_noise(BAProblem(cams, pts, None), *SIN, ctx=ctx)
    assert np.allclose(out.cameras, oc, rtol=RTOL, atol=ATOL)
    assert np.allclose(out.points, op, rtol=RTOL, atol=ATOL)
    rp = ResidentProblem(ctx)
    rp.upload_points(pts)
    rp.upload_cameras(cams)
    rp.add_sin_noise(*SIN)
    rc, rpts = rp.download_problem(C, len(pts))
    assert bits_equal(rc, out.cameras) and bits_equal(rpts, out.points)


# ---- full-size workloads ----------------------------------------------------------------------------------------
_WORKLOADS = {}


def workload(c2b, ctx, name):
    """(cams, pts, scene, graph of a resident pass) of a BASELINE config, built once per module"""
    if name not in _WORKLOADS:
        import bench
        from city2ba_b200.generate import ResidentProblem
        _WORKLOADS.clear()                                       # one at a time: cfg4 holds a few GB
        cams, pts, xyz, tri = bench.build_workload(name)
        scene = c2b.Scene(xyz, tri, ctx=ctx)
        rp = ResidentProblem(ctx)
        rp.upload_points(pts)
        rp.upload_cameras(cams)
        rp.run(scene, bench.MAX_DIST)
        _WORKLOADS[name] = (cams, pts, scene, rp.download())
    return _WORKLOADS[name]


@pytest.fixture(scope="module", autouse=True)
def _drop_workloads():
    yield
    _WORKLOADS.clear()


# ---- resident reprojection error -------------------------------------------------------------------------------
NORMS = [1.0, 2.0, 0.5, 1.5, 3.0]
FAR = cams_at([[1e5, 1e5, 1e5]])[0]                             # farther than max_dist from every point


def with_empty_runs(cams):
    """runs of cameras without observations at the start, in the middle and at the end of the camera array"""
    h = len(cams) // 2
    return np.concatenate([np.tile(FAR, (3, 1)), cams[:h], np.tile(FAR, (5, 1)), cams[h:], np.tile(FAR, (4, 1))])


def projected_terms(cams, pts, offsets, point_idx, uv, norm):
    """|q - uv|^p summed per observation, q from the host mirror's _project_all, in camera ranges of ~2 M obs"""
    from city2ba_b200.baproblem import _project_all
    off = np.asarray(offsets, np.uint64)
    out = np.empty(len(uv))
    c0 = 0
    while c0 < len(cams):
        c1 = min(len(cams), int(np.searchsorted(off, off[c0] + 2_000_000, side="right")) - 1)
        c1 = max(c1, c0 + 1)
        o0, o1 = int(off[c0]), int(off[c1])
        if o1 > o0:
            q = _project_all(cams[c0:c1], pts, off[c0:c1 + 1] - off[c0], point_idx[o0:o1])
            d = np.abs(q - uv[o0:o1])
            out[o0:o1] = (d ** norm).sum(axis=1) if norm != 2.0 else (d * d).sum(axis=1)
        c0 = c1
    return out


def check_reproj(got, terms, norm):
    ref, tol, tol_sum = reproj_tolerance(terms, norm)
    assert abs(got - ref) <= tol, (norm, got, ref, tol)
    # the terms are random and a few lie near zero: dropping or doubling any but the smallest tenth of them moves
    # the result past the tolerance
    assert tol_sum < np.quantile(terms, 0.1)


@pytest.mark.parametrize("size", ["below", "above", "cfg3", "cfg4"])
def test_reprojection_error_resident(c2b, ctx, size):
    import bench
    from city2ba_b200.generate import ResidentProblem
    cams, pts, scene, g = workload(c2b, ctx, "cfg4" if size == "cfg4" else "cfg3")
    if size in ("below", "above"):
        off = g.offsets
        k = int(np.searchsorted(off, THREADS)) - 1 if size == "below" else int(np.searchsorted(off, THREADS, "right"))
        cams = cams[:k]
    cams = with_empty_runs(cams)
    rp = ResidentProblem(ctx)
    rp.upload_points(pts)
    rp.upload_cameras(cams)
    rp.run(scene, bench.MAX_DIST)
    g0 = rp.download()
    O = g0.num_observations
    counts = np.diff(g0.offsets.astype(np.int64))
    assert np.all(counts[np.all(cams == FAR, axis=1)] == 0) and O > 0
    if size == "below":
        assert THREADS - 20_000 < O < THREADS
    elif size == "above":
        assert THREADS < O < THREADS + 20_000
    # un-noised: the visibility pass and k_reproj_partial project with the same round-to-nearest operations
    for p in NORMS:
        assert rp.reprojection_error(p) == 0.0, p
    # observation noise only: the terms are |uv0 - uv1|^p of the CSR before and after
    rp.add_noise(0.0, 0.0, 0.0, 1e-2, seed=3)
    g1 = rp.download()
    assert np.array_equal(g1.offsets, g0.offsets) and np.array_equal(g1.point_idx, g0.point_idx)
    d = np.abs(g0.uv - g1.uv)
    for p in NORMS:
        check_reproj(rp.reprojection_error(p), (d * d).sum(axis=1) if p == 2.0 else (d ** p).sum(axis=1), p)
    del d
    # camera and point noise: the terms of the host mirror's projection of the downloaded problem
    rp.add_noise(1e-5, 1e-4, 1e-3, 0.0, seed=4)
    rc, rpts = rp.download_problem(len(cams), len(pts))
    for p in NORMS:
        check_reproj(rp.reprojection_error(p), projected_terms(rc, rpts, g0.offsets, g0.point_idx, g1.uv, p), p)


# ---- resident vs host entry vs oracle at full size ----------------------------------------------------------------
def _ops():
    return {
        "drift_normalized": (lambda rp: rp.add_drift(1e-3, 0.1, 0.2, None, seed=11),
                             lambda c2b, ba, ctx: c2b.noise.add_drift_normalized(ba, 1e-3, 0.1, 0.2, seed=11, ctx=ctx),
                             lambda orc, c, p, uv: orc.add_drift_normalized(c, p, 1e-3, 0.1, 0.2, 11) + (uv,)),
        "drift_dir": (lambda rp: rp.add_drift(2e-3, 0.1, 0.2, DRIFT_DIR, seed=12),
                      lambda c2b, ba, ctx: c2b.noise.add_drift(ba, 2e-3, 0.1, 0.2, DRIFT_DIR, seed=12, ctx=ctx),
                      lambda orc, c, p, uv: orc.add_drift(c, p, 2e-3, 0.1, 0.2, DRIFT_DIR, 12) + (uv,)),
        **{f"noise_pt{ps}_obs{os_}": (
            lambda rp, ps=ps, os_=os_: rp.add_noise(1e-3, 1e-4, ps, os_, seed=13),
            lambda c2b, ba, ctx, ps=ps, os_=os_: c2b.noise.add_noise(ba, 1e-3, 1e-4, ps, os_, seed=13, ctx=ctx),
            lambda orc, c, p, uv, ps=ps, os_=os_: orc.add_noise(c, p, uv, 1e-3, 1e-4, ps, os_, 13))
            for ps in (0.0, 1e-3) for os_ in (0.0, 1e-3)},
        "sin": (lambda rp: rp.add_sin_noise(*SIN),
                lambda c2b, ba, ctx: c2b.noise.add_sin_noise(ba, *SIN, ctx=ctx),
                lambda orc, c, p, uv: orc.add_sin_noise(c, p, *SIN) + (uv,)),
    }


OPS = _ops()
# the arrays the oracle reproduces bit for bit (test_gpu_noise.py); the rest to RTOL
EXACT = {"drift_dir": ("pts",), **{k: ("pts", "uv") for k in OPS if k.startswith("noise")}}


def run_op(c2b, orc, ctx, cams, pts, scene, g0, name):
    import bench
    from city2ba_b200.baproblem import BAProblem
    from city2ba_b200.generate import ResidentProblem, VisGraph
    res, host, ref = OPS[name]
    rp = ResidentProblem(ctx)
    rp.upload_points(pts)
    rp.upload_cameras(cams)
    rp.run(scene, bench.MAX_DIST)
    res(rp)
    rc, rpts = rp.download_problem(len(cams), len(pts))
    ruv = rp.download().uv
    h = host(c2b, BAProblem(cams, pts, VisGraph(g0.offsets, g0.point_idx, g0.uv)), ctx)
    assert bits_equal(rc, h.cameras) and bits_equal(rpts, h.points) and bits_equal(ruv, h.vis_graph.uv)
    oc, op, ouv = ref(orc, cams, pts, g0.uv)
    assert np.allclose(rc, oc, rtol=RTOL, atol=ATOL)
    exact = EXACT.get(name, ())
    # (array_equal: where a standard deviation is 0 the GPU skips the array and the oracle adds +-0, which can
    # turn a -0.0 into +0.0)
    assert np.array_equal(rpts, op) if "pts" in exact else np.allclose(rpts, op, rtol=RTOL, atol=ATOL)
    assert np.array_equal(ruv, ouv) if "uv" in exact else np.allclose(ruv, ouv, rtol=RTOL, atol=ATOL)
    return rp, rc, rpts


@pytest.mark.parametrize("cfg,name", [("cfg3", k) for k in OPS] +
                         [("cfg4", "noise_pt0.001_obs0.001"), ("cfg4", "drift_normalized")])
def test_resident_host_oracle_full_size(c2b, orc, ctx, cfg, name):
    cams, pts, scene, g0 = workload(c2b, ctx, cfg)
    run_op(c2b, orc, ctx, cams, pts, scene, g0, name)


@pytest.mark.parametrize("name", list(OPS))
def test_visibility_after_resident_noise(c2b, orc, ctx, name):
    """after each op, a new resident pass sees the noised problem: the oracle's graph of the downloaded arrays"""
    cams, pts = orc.grid_cameras(10, 4), orc.grid_points(10, 4)
    xyz, tri = orc.city_mesh(4)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    from city2ba_b200.generate import ResidentProblem
    rp = ResidentProblem(ctx)
    rp.upload_points(pts)
    rp.upload_cameras(cams)
    rp.run(scene, 10.0)
    g0 = rp.download()
    rp, rc, rpts = run_op(c2b, orc, ctx, cams, pts, scene, g0, name)
    rp.run(scene, 10.0)
    assert_same_graph(rp.download(), orc.visibility_graph(xyz, tri, rc, rpts, 10.0), name)


# ---- c2b_add_noise streams the observations in chunks of max(2^20, ceil(O / 16)) ----------------------------------
@pytest.mark.parametrize("O", [2 ** 20 - 1, 2 ** 20, 2 ** 20 + 1, 2 * 2 ** 20 + 1, 16 * 2 ** 20 + 17])
def test_add_noise_streaming_boundaries(c2b, orc, ctx, O):
    cams = cams_at([[0.0, 0.0, 0.0], [1.0, 2.0, 3.0]])
    pts = np.arange(9.0).reshape(3, 3)
    uv = np.random.default_rng(O).uniform(-1.0, 1.0, (O, 2))
    uv[::7] = -0.0                                               # the sign of zero is part of the result
    g = c2b.VisGraph(np.array([0, O // 2, O], np.uint64), np.zeros(O, np.uint64), uv)
    out = c2b.noise.add_noise(c2b.BAProblem(cams, pts, g), 0.0, 0.0, 0.0, 0.01, seed=21, ctx=ctx)
    _, _, ouv = orc.add_noise(cams, pts, uv, 0.0, 0.0, 0.0, 0.01, 21)
    assert bits_equal(out.vis_graph.uv, ouv)
    assert not np.array_equal(ouv, uv)
