"""The test suite's CPU restatement of the GPU's add_incorrect_correspondences rule (tests/mismatch_ref.c), without a
GPU: its draws are Philox4x32-10's, its picks follow the reference's weights (maxd - d_j, maxd for the observation
itself), its selections the chance, and its errors Rng::weighted's.  tests/test_gpu_mismatch.py compares the GPU
entries with it bit for bit through the `mm_ref` fixture defined here."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

from conftest import ROOT


class MismatchRef:
    """ctypes binding of tests/mismatch_ref.c, compiled into `out_dir` (the checkout may be read-only)"""

    def __init__(self, out_dir):
        so = os.path.join(str(out_dir), "libmismatch_ref.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                               "-Wextra", "-shared", "-o", so, os.path.join(ROOT, "tests", "mismatch_ref.c"), "-lm"])
        self.lib = C.CDLL(so)
        self.lib.mm_add_incorrect_correspondences.restype = C.c_int

    def philox4x32_10(self, ctr, key):
        ctr = np.ascontiguousarray(ctr, np.uint32)
        key = np.ascontiguousarray(key, np.uint32)
        out = np.empty(4, np.uint32)
        p32 = C.POINTER(C.c_uint32)
        self.lib.mm_philox4x32_10(ctr.ctypes.data_as(p32), key.ctypes.data_as(p32), out.ctypes.data_as(p32))
        return out

    def add_incorrect_correspondences(self, offsets, point_idx, uv, mismatch_chance, seed, want_picks=False):
        """(point_idx u32, stats dict n_selected / n_swapped, error None | ("AllWeightsZero" | "NegativeWeight",
        observation)) and, with want_picks, the partner of every observation (-1 when not selected).  point_idx is
        unchanged on an error."""
        off = np.ascontiguousarray(offsets, np.uint64)
        idx = np.ascontiguousarray(point_idx, np.uint32).copy()
        uv = np.ascontiguousarray(uv, np.float64).reshape(-1)
        picks = np.empty(int(off[-1]), np.int64) if want_picks else None
        ns, nw, eo = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        rc = self.lib.mm_add_incorrect_correspondences(
            off.ctypes.data_as(C.POINTER(C.c_uint64)), C.c_uint64(len(off) - 1),
            idx.ctypes.data_as(C.POINTER(C.c_uint32)), uv.ctypes.data_as(C.POINTER(C.c_double)),
            C.c_double(mismatch_chance), C.c_uint64(int(seed) & (2 ** 64 - 1)), C.byref(ns), C.byref(nw),
            picks.ctypes.data_as(C.POINTER(C.c_int64)) if want_picks else None, C.byref(eo))
        err = None if rc == 0 else ({1: "AllWeightsZero", 2: "NegativeWeight"}[rc], int(eo.value))
        out = (idx, {"n_selected": int(ns.value), "n_swapped": int(nw.value)}, err)
        return out + (picks,) if want_picks else out


@pytest.fixture(scope="session")
def mm_ref(tmp_path_factory):
    return MismatchRef(tmp_path_factory.mktemp("mismatch_ref"))


def test_philox_is_the_noise_stream(mm_ref, orc):
    """the restatement's Philox4x32-10 is the one the noise pass's checker uses"""
    rng = np.random.default_rng(8)
    for _ in range(50):
        ctr, key = rng.integers(0, 2 ** 32, 4, dtype=np.uint64), rng.integers(0, 2 ** 32, 2, dtype=np.uint64)
        assert np.array_equal(mm_ref.philox4x32_10(ctr, key), orc.philox4x32_10(ctr, key))


def _cameras(n_cams, uv_cam):
    """n_cams identical cameras, each holding the observations uv_cam"""
    k = len(uv_cam)
    off = np.arange(n_cams + 1, dtype=np.uint64) * k
    idx = np.arange(n_cams * k, dtype=np.uint32)
    return off, idx, np.tile(np.asarray(uv_cam, np.float64), (n_cams, 1))


def test_picks_follow_unquantised_weights(mm_ref):
    uv_cam = [(0.0, 0.0), (1.0, 0.0), (3.0, 1.0), (-2.0, 4.0), (5.5, -1.5), (0.5, 0.25), (-4.0, -3.0), (2.0, 7.0)]
    k, n_cams = len(uv_cam), 4000
    off, idx, uv = _cameras(n_cams, uv_cam)
    out, st, err, picks = mm_ref.add_incorrect_correspondences(off, idx, uv, 1.0, 2024, want_picks=True)
    assert err is None and st["n_selected"] == n_cams * k
    local = picks.reshape(n_cams, k) - (np.arange(n_cams, dtype=np.int64) * k)[:, None]
    assert local.min() >= 0 and local.max() < k
    p = np.asarray(uv_cam)
    d = np.sqrt(((p[:, None, :] - p[None, :, :]) ** 2).sum(axis=2))
    pvals = []
    for i in range(k):
        w = d[i].max() - d[i]
        w[i] = d[i].max()
        expected = w / w.sum() * n_cams
        observed = np.bincount(local[:, i], minlength=k)
        assert observed[w == 0].sum() == 0, "a zero-weight partner was picked"
        keep = w > 0
        pvals.append(stats.chisquare(observed[keep], expected[keep]).pvalue)
    # eight tests: Bonferroni at 1e-3 overall
    assert min(pvals) > 1e-3 / k, pvals
    # the swaps: n_swapped counts the picks of another observation, the result is the transpositions in order
    assert st["n_swapped"] == int(np.sum(local != np.arange(k)[None, :]))
    ref = idx.copy()
    for o in range(len(idx)):
        j = picks[o]
        ref[o], ref[j] = ref[j], ref[o]
    assert np.array_equal(out, ref)


def test_selected_fraction(mm_ref):
    rng = np.random.default_rng(5)
    counts = rng.integers(0, 40, 3000)
    off = np.zeros(len(counts) + 1, np.uint64)
    off[1:] = np.cumsum(counts)
    O = int(off[-1])
    _, st, err = mm_ref.add_incorrect_correspondences(off, np.zeros(O, np.uint32), rng.normal(size=(O, 2)), 0.3, 11)
    assert err is None
    n = int(counts[counts > 1].sum())
    sd = np.sqrt(n * 0.3 * 0.7)
    assert abs(st["n_selected"] - 0.3 * n) < 5 * sd


@pytest.mark.parametrize("kind", ["AllWeightsZero", "NegativeWeight"])
def test_errors(mm_ref, kind):
    rng = np.random.default_rng(6)
    off = np.array([0, 3, 4, 9], np.uint64)
    idx = np.arange(9, dtype=np.uint32)
    uv = rng.normal(size=(9, 2))
    uv[3] = np.nan                      # camera 1 has one observation: never drawn from
    if kind == "AllWeightsZero":
        uv[4:9] = uv[4]                 # camera 2: coinciding observations
    else:
        uv[6] = (np.nan, 0.0)
    out, st, err = mm_ref.add_incorrect_correspondences(off, idx, uv, 1.0, 1)
    assert err == (kind, 4)             # the first selected observation of camera 2
    assert np.array_equal(out, idx)     # unchanged
    # no error when the failing camera has no selected observation
    for p in (0.0, float("nan")):
        out, st, err = mm_ref.add_incorrect_correspondences(off, idx, uv, p, 1)
        assert err is None and st["n_selected"] == 0 and np.array_equal(out, idx)
    ok = uv.copy()
    ok[4:9] = rng.normal(size=(5, 2))
    _, st, err = mm_ref.add_incorrect_correspondences(off, idx, ok, 1.0, 1)
    assert err is None and st["n_selected"] == 8


def test_deterministic_and_empty(mm_ref):
    rng = np.random.default_rng(7)
    off = np.array([0, 10, 10, 30], np.uint64)
    uv = rng.normal(size=(30, 2))
    a = mm_ref.add_incorrect_correspondences(off, np.arange(30), uv, 0.5, 3)
    b = mm_ref.add_incorrect_correspondences(off, np.arange(30), uv, 0.5, 3)
    c = mm_ref.add_incorrect_correspondences(off, np.arange(30), uv, 0.5, 4)
    assert np.array_equal(a[0], b[0]) and a[1] == b[1]
    assert not np.array_equal(a[0], c[0])
    for off in (np.zeros(1, np.uint64), np.zeros(3, np.uint64)):
        out, st, err = mm_ref.add_incorrect_correspondences(off, np.zeros(0), np.zeros((0, 2)), 1.0, 3)
        assert err is None and len(out) == 0 and st == {"n_selected": 0, "n_swapped": 0}
