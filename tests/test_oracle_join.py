"""The test suite's CPU restatement of the GPU's join_landmarks rule (tests/join_ref.c), without a GPU: its draws are
Philox4x32-10's, its selections an exact-size uniform subset, its picks uniform over the 10 neighbours, its neighbours
those of a k-d tree, and its errors the host forms'.  tests/test_gpu_join.py compares the GPU entries with it bit for
bit through the `jn_ref` fixture defined here."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats
from scipy.spatial import cKDTree

from conftest import ROOT

U32P, U64P, DP = C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_double)


class JoinRef:
    """ctypes binding of tests/join_ref.c, compiled into `out_dir` (the checkout may be read-only)"""

    def __init__(self, out_dir):
        so = os.path.join(str(out_dir), "libjoin_ref.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                               "-Wextra", "-shared", "-o", so, os.path.join(ROOT, "tests", "join_ref.c"), "-lm"])
        self.lib = C.CDLL(so)
        self.lib.jn_join_landmarks.restype = C.c_int
        self.lib.jn_neighbours.restype = C.c_uint64
        self.lib.jn_count.restype = C.c_uint64
        self.lib.jn_count.argtypes = [C.c_double, C.c_uint64, C.c_uint64]

    def philox4x32_10(self, ctr, key):
        ctr = np.ascontiguousarray(ctr, np.uint32)
        key = np.ascontiguousarray(key, np.uint32)
        out = np.empty(4, np.uint32)
        self.lib.jn_philox4x32_10(ctr.ctypes.data_as(U32P), key.ctypes.data_as(U32P), out.ctypes.data_as(U32P))
        return out

    def count(self, join_percent, P, O):
        return int(self.lib.jn_count(float(join_percent), int(P), int(O)))

    def neighbours(self, pts, q):
        """the m = min(11, P) smallest (d2, index) pairs of point q: (indices, d2)"""
        pts = np.ascontiguousarray(pts, np.float64).reshape(-1, 3)
        nb, d2 = np.empty(11, np.uint32), np.empty(11)
        m = self.lib.jn_neighbours(pts.ctypes.data_as(DP), C.c_uint64(len(pts)), C.c_uint64(int(q)),
                                   nb.ctypes.data_as(U32P), d2.ctypes.data_as(DP))
        return nb[:m], d2[:m]

    def join_landmarks(self, pts, point_idx, join_percent, seed, want_selected=False):
        """(point_idx u32, stats dict n_selected / n_changed, error None | "No neighbors?!" | ("not finite", point))
        and, with want_selected, the selection mask.  point_idx is unchanged on an error."""
        pts = np.ascontiguousarray(pts, np.float64).reshape(-1, 3)
        idx = np.ascontiguousarray(point_idx, np.uint32).copy()
        sel = np.zeros(max(len(idx), 1), np.uint8)
        ns, nc, bad = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        rc = self.lib.jn_join_landmarks(pts.ctypes.data_as(DP), C.c_uint64(len(pts)), idx.ctypes.data_as(U32P),
                                        C.c_uint64(len(idx)), C.c_double(join_percent),
                                        C.c_uint64(int(seed) & (2 ** 64 - 1)), C.byref(ns), C.byref(nc),
                                        sel.ctypes.data_as(C.POINTER(C.c_uint8)), C.byref(bad))
        err = {0: None, 1: "No neighbors?!", 2: ("not finite", int(bad.value))}[rc]
        out = (idx, {"n_selected": int(ns.value), "n_changed": int(nc.value)}, err)
        return out + (sel[:len(idx)].astype(bool),) if want_selected else out


@pytest.fixture(scope="session")
def jn_ref(tmp_path_factory):
    return JoinRef(tmp_path_factory.mktemp("join_ref"))


def test_philox_is_the_noise_stream(jn_ref, orc):
    """the restatement's Philox4x32-10 is the one the noise pass's checker uses"""
    rng = np.random.default_rng(9)
    for _ in range(50):
        ctr, key = rng.integers(0, 2 ** 32, 4, dtype=np.uint64), rng.integers(0, 2 ** 32, 2, dtype=np.uint64)
        assert np.array_equal(jn_ref.philox4x32_10(ctr, key), orc.philox4x32_10(ctr, key))


def test_selection_count_and_uniformity(jn_ref):
    rng = np.random.default_rng(10)
    pts = rng.normal(size=(40, 3))
    O = 60
    idx = rng.integers(0, 40, O).astype(np.uint32)
    # exact count: min(floor(join_percent P), O)
    for jp, want in ((0.0, 0), (-1.0, 0), (float("nan"), 0), (0.024, 0), (0.025, 1), (0.5, 20), (1.0, 40),
                     (1.5, 60), (100.0, 60)):
        _, st, err, sel = jn_ref.join_landmarks(pts, idx, jp, 3, want_selected=True)
        assert err is None and st["n_selected"] == want == int(sel.sum()) == jn_ref.count(jp, 40, O), jp
    # every position is selected with probability k / O
    seeds = 3000
    hits = np.zeros(O)
    for s in range(seeds):
        _, st, _, sel = jn_ref.join_landmarks(pts, idx, 0.25, s, want_selected=True)  # k = 10
        assert st["n_selected"] == 10
        hits += sel
    assert stats.chisquare(hits, np.full(O, seeds * 10 / O)).pvalue > 1e-3


def test_picks_uniform_over_ten_neighbours(jn_ref):
    rng = np.random.default_rng(11)
    P, O = 30, 30000
    pts = rng.normal(size=(P, 3))
    idx = rng.integers(0, P, O).astype(np.uint32)
    out, st, err = jn_ref.join_landmarks(pts, idx, O / P + 1.0, 12)
    assert err is None and st["n_selected"] == O
    lists = [jn_ref.neighbours(pts, q)[0] for q in range(P)]
    at = np.array([int(np.nonzero(lists[q] == p)[0][0]) for q, p in zip(idx, out)])
    assert at.min() >= 1 and at.max() <= 10        # never the point itself (distinct points), one of the next 10
    assert st["n_changed"] == O
    counts = np.bincount(at, minlength=11)[1:]
    assert stats.chisquare(counts, np.full(10, O / 10)).pvalue > 1e-3


def test_neighbours_equal_kd_tree(jn_ref):
    rng = np.random.default_rng(12)
    for P in (2, 5, 11, 12, 500):
        pts = rng.uniform(-50, 50, size=(P, 3))
        tree = cKDTree(pts)
        for q in range(0, P, max(1, P // 40)):
            nb, d2 = jn_ref.neighbours(pts, q)
            d, near = tree.query(pts[q], k=min(11, P))
            assert np.array_equal(nb, np.atleast_1d(near)), (P, q)
            assert np.allclose(d2, np.atleast_1d(d) ** 2, rtol=1e-12, atol=0)
            assert nb[0] == q


def test_coincident_points_order_by_index(jn_ref):
    pts = np.zeros((14, 3))
    pts[12:] = 5.0
    nb, d2 = jn_ref.neighbours(pts, 7)
    assert list(nb) == list(range(11)) and not d2.any()     # q = 7 is not first: 0..10 by index
    # q can pick itself: over many seeds, the picks of observations of point 7 include 7
    idx = np.full(200, 7, np.uint32)
    out, st, err = jn_ref.join_landmarks(pts, idx, 200 / 14 + 1, 1)
    assert err is None and st["n_selected"] == 200 and 0 < st["n_changed"] < 200
    assert set(out.tolist()) == set(range(1, 11))


def test_errors(jn_ref):
    idx = np.zeros(5, np.uint32)
    out, st, err = jn_ref.join_landmarks(np.ones((1, 3)), idx, 1.0, 1)
    assert err == "No neighbors?!" and np.array_equal(out, idx)
    # nothing selected: no error (n = floor(0.5 * 1) = 0, or no observations)
    assert jn_ref.join_landmarks(np.ones((1, 3)), idx, 0.5, 1)[2] is None
    assert jn_ref.join_landmarks(np.ones((1, 3)), idx[:0], 1.0, 1)[2] is None
    rng = np.random.default_rng(13)
    pts = rng.normal(size=(20, 3))
    idx = rng.integers(0, 20, 30).astype(np.uint32)
    for bad in (np.nan, np.inf, -np.inf):
        p = pts.copy()
        p[13, 2] = bad
        p[17, 0] = bad
        out, st, err = jn_ref.join_landmarks(p, idx, 0.5, 1)
        assert err == ("not finite", 13) and np.array_equal(out, idx)
        assert jn_ref.join_landmarks(p, idx, 0.0, 1)[2] is None
    # coordinates near 1e154: d2 overflows to inf, still a total order by index
    big = rng.normal(size=(15, 3)) * 1e154
    out, st, err = jn_ref.join_landmarks(big, rng.integers(0, 15, 40), 1.0, 2)
    assert err is None and st["n_selected"] == 15
    assert np.isinf(jn_ref.neighbours(big, 0)[1]).any()
