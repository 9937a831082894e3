"""Host mirror of city2ba::noise for the elementwise passes (reference: src/noise.rs:35-177).

The reference draws from rand's thread_rng(), which cannot be seeded; here every function takes
a `seed` for the Philox4x32-10 stream (default: a fresh 64-bit seed from os.urandom, i.e. the
reference's "different every run" behaviour).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from ._lib import check, context, lib
from .baproblem import BAProblem
from .generate import VisGraph

_pd = C.POINTER(C.c_double)


def _seed(seed):
    return int.from_bytes(os.urandom(8), "little") if seed is None else int(seed) & (2 ** 64 - 1)


def _p(a):
    return a.ctypes.data_as(_pd)


def add_drift(bal: BAProblem, strength, angle_strength, std, dir, seed=None, ctx=None) -> BAProblem:
    """src/noise.rs:68-116"""
    ctx = ctx or context()
    cams, pts = bal.cameras.copy(), bal.points.copy()
    d = np.ascontiguousarray(dir, np.float64)
    check(lib().c2b_add_drift(ctx.handle, _p(cams), len(cams), _p(pts), len(pts), float(strength),
                              float(angle_strength), float(std), _p(d), _seed(seed)))
    return BAProblem(cams, pts, bal.vis_graph)


def add_drift_normalized(bal: BAProblem, strength, angle_strength, std, seed=None, ctx=None) -> BAProblem:
    """src/noise.rs:47-56"""
    ctx = ctx or context()
    cams, pts = bal.cameras.copy(), bal.points.copy()
    check(lib().c2b_add_drift_normalized(ctx.handle, _p(cams), len(cams), _p(pts), len(pts),
                                         float(strength), float(angle_strength), float(std),
                                         _seed(seed)))
    return BAProblem(cams, pts, bal.vis_graph)


def add_noise(bal: BAProblem, translation_std, rotation_std, point_std, observations_std,
              seed=None, ctx=None) -> BAProblem:
    """src/noise.rs:119-177"""
    ctx = ctx or context()
    cams, pts = bal.cameras.copy(), bal.points.copy()
    g = bal.vis_graph
    uv = np.ascontiguousarray(g.uv, np.float64).copy()
    check(lib().c2b_add_noise(ctx.handle, _p(cams), len(cams), _p(pts), len(pts), _p(uv), len(uv),
                              float(translation_std), float(rotation_std), float(point_std),
                              float(observations_std), _seed(seed)))
    return BAProblem(cams, pts, VisGraph(g.offsets, g.point_idx, uv))


def add_sin_noise(bal: BAProblem, dir, noise_dir, strength, frequency, ctx=None) -> BAProblem:
    """src/noise.rs:388-416"""
    ctx = ctx or context()
    cams, pts = bal.cameras.copy(), bal.points.copy()
    d = np.ascontiguousarray(dir, np.float64)
    nd = np.ascontiguousarray(noise_dir, np.float64)
    check(lib().c2b_add_sin_noise(ctx.handle, _p(cams), len(cams), _p(pts), len(pts), _p(d), _p(nd),
                                  float(strength), float(frequency)))
    return BAProblem(cams, pts, bal.vis_graph)


def last_timing(ctx=None):
    """device milliseconds of the last noise call: (upload, statistics + kernels, download)"""
    ctx = ctx or context()
    ms = (C.c_float * 3)()
    check(lib().c2b_noise_timing(ctx.handle, ms))
    return tuple(float(x) for x in ms)


# ---- graph-editing noise (src/noise.rs:180-378): sequential, data-dependent edits of the observation graph,
# host side like the reference's; the same procedures as include/city2ba.hpp.  Seeded (numpy Generator);
# parity with the reference's thread_rng() draws is distributional.

def _with_graph(bal: BAProblem, offsets, idx, uv, points=None) -> BAProblem:
    return BAProblem(bal.cameras.copy(), bal.points.copy() if points is None else points,
                     VisGraph(np.asarray(offsets, np.uint64), np.asarray(idx, np.uint64), np.asarray(uv, np.float64)))


def add_incorrect_correspondences(bal: BAProblem, mismatch_chance, seed=None) -> BAProblem:
    """src/noise.rs:180-226: with probability mismatch_chance an observation trades its point index with another
    observation of the same camera, chosen with weight (largest image distance) - (its image distance) — as
    written there, which also gives the observation itself the largest weight"""
    rng = np.random.default_rng(seed)
    g = bal.vis_graph
    idx = g.point_idx.copy()
    off = g.offsets.astype(np.int64)
    for c in range(len(g)):
        a, b = off[c], off[c + 1]
        if b - a <= 1:
            continue
        uv = g.uv[a:b]
        for i in np.nonzero(rng.uniform(size=b - a) <= mismatch_chance)[0]:
            w = -np.sqrt(((uv - uv[i]) ** 2).sum(axis=1))
            w[i] = 0.0
            w = w - w.min()
            if not w.sum() > 0:
                raise AssertionError("called `Result::unwrap()` on an `Err` value: AllWeightsZero")
            j = rng.choice(b - a, p=w / w.sum())
            idx[a + i], idx[a + j] = idx[a + j], idx[a + i]
    return _with_graph(bal, g.offsets, idx, g.uv)


def _weight_error(e):
    """C2BError of a selection with invalid weights -> the host form's AssertionError (same message tail)"""
    from ._lib import ERR_INVALID, C2BError
    if isinstance(e, C2BError) and e.code == ERR_INVALID and "called `Result::unwrap()` on an `Err` value" in str(e):
        return AssertionError(str(e))
    return None


def add_incorrect_correspondences_gpu(bal: BAProblem, mismatch_chance, seed=None, ctx=None, stats=None) -> BAProblem:
    """add_incorrect_correspondences on the GPU (c2b_add_incorrect_correspondences): the same operation with the
    library's deterministic draws, a pure function of `seed` (default: a fresh one from os.urandom), so it does not
    reproduce the numpy draws of the host form.  Raises AssertionError on a selected observation whose image distances
    are all 0 (AllWeightsZero) or not all finite (NegativeWeight).  Works on copies; `stats`, a dict if given, receives
    the call's c2b_mismatch_stats (n_selected, n_swapped, device times)."""
    from ._lib import C2BError, MismatchStats
    ctx = ctx or context()
    g = bal.vis_graph
    off = np.array(g.offsets, np.uint64, order="C")
    if len(off) != len(bal.cameras) + 1:
        raise ValueError("cameras and CSR offsets disagree")
    idx = g.point_idx
    if len(idx) and int(idx.max()) > 0xffffffff:
        raise ValueError("point index does not fit 32 bits")
    idx = np.array(idx, np.uint32, order="C")
    uv = np.array(g.uv, np.float64, order="C").reshape(-1, 2)
    st = MismatchStats()
    try:
        check(lib().c2b_add_incorrect_correspondences(ctx.handle, off.ctypes.data_as(C.POINTER(C.c_uint64)),
                                                      len(off) - 1, idx.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                      _p(uv), float(mismatch_chance), _seed(seed), C.byref(st)))
    except C2BError as e:
        a = _weight_error(e)
        if a is not None:
            raise a from e
        raise
    if stats is not None:
        stats.update(st.to_dict())
    return _with_graph(bal, off, idx, uv)


def _no_neighbors(e):
    """C2BError of a join with fewer than two points -> the host form's AssertionError (same message tail)"""
    from ._lib import ERR_INVALID, C2BError
    if isinstance(e, C2BError) and e.code == ERR_INVALID and str(e).endswith("No neighbors?!"):
        return AssertionError(str(e))
    return None


def join_landmarks_gpu(bal: BAProblem, join_percent, seed=None, ctx=None, stats=None) -> BAProblem:
    """join_landmarks on the GPU (c2b_join_landmarks): the same operation with the library's deterministic draws, a
    pure function of `seed` (default: a fresh one from os.urandom), so it does not reproduce the numpy draws of the
    host form.  The 10 neighbours are exact: the 11 nearest points by (squared distance, index), the first skipped.
    Raises AssertionError ("No neighbors?!") when observations are selected among fewer than two points, and
    C2BError when a point is not finite.  Works on copies; `stats`, a dict if given, receives the call's
    c2b_join_stats (n_selected, n_changed, device times)."""
    from ._lib import C2BError, JoinStats
    ctx = ctx or context()
    g = bal.vis_graph
    off = np.array(g.offsets, np.uint64, order="C")
    if len(off) != len(bal.cameras) + 1:
        raise ValueError("cameras and CSR offsets disagree")
    idx = g.point_idx
    if len(idx) and int(idx.max()) > 0xffffffff:
        raise ValueError("point index does not fit 32 bits")
    idx = np.array(idx, np.uint32, order="C")
    pts = np.array(bal.points, np.float64, order="C").reshape(-1, 3)
    st = JoinStats()
    try:
        check(lib().c2b_join_landmarks(ctx.handle, _p(pts), len(pts), off.ctypes.data_as(C.POINTER(C.c_uint64)),
                                       len(off) - 1, idx.ctypes.data_as(C.POINTER(C.c_uint32)), float(join_percent),
                                       _seed(seed), C.byref(st)))
    except C2BError as e:
        a = _no_neighbors(e)
        if a is not None:
            raise a from e
        raise
    if stats is not None:
        stats.update(st.to_dict())
    return _with_graph(bal, off, idx, g.uv)


def drop_features(bal: BAProblem, drop_percent, seed=None) -> BAProblem:
    """src/noise.rs:229-250: every camera keeps floor(len * drop_percent) of its observations, chosen by a shuffle"""
    rng = np.random.default_rng(seed)
    g = bal.vis_graph
    off = g.offsets.astype(np.int64)
    keep, counts = [], []
    for c in range(len(g)):
        a, b = off[c], off[c + 1]
        perm = a + rng.permutation(b - a)
        k = min(int((b - a) * drop_percent), b - a)
        keep.append(perm[:k])
        counts.append(k)
    keep = np.concatenate(keep) if keep else np.zeros(0, np.int64)
    return _with_graph(bal, np.concatenate([[0], np.cumsum(counts)]), g.point_idx[keep], g.uv[keep])


def split_landmarks(bal: BAProblem, split_percent, seed=None) -> BAProblem:
    """src/noise.rs:254-288: floor(split_percent * points) landmarks get a copy at the same location; each of
    their observations moves to the copy with probability 1/2"""
    rng = np.random.default_rng(seed)
    g = bal.vis_graph
    l = len(bal.points)
    n = int(split_percent * l)
    inds = rng.choice(l, size=n, replace=False)
    target = np.full(l, -1, np.int64)
    target[inds] = l + np.arange(n)
    idx = g.point_idx.astype(np.int64).copy()
    move = (target[idx] >= 0) & (rng.uniform(size=len(idx)) < 0.5)
    idx[move] = target[idx[move]]
    return _with_graph(bal, g.offsets, idx, g.uv, points=np.concatenate([bal.points, bal.points[inds]]))


def join_landmarks(bal: BAProblem, join_percent, seed=None) -> BAProblem:
    """src/noise.rs:323-378: floor(join_percent * points) observations (drawn over ALL observations) are
    re-pointed at one of the 10 nearest other landmarks of the landmark they see"""
    from scipy.spatial import cKDTree
    rng = np.random.default_rng(seed)
    g = bal.vis_graph
    n = int(join_percent * len(bal.points))
    idx = g.point_idx.astype(np.int64).copy()
    if n and len(idx):
        if len(bal.points) < 2:
            raise AssertionError("No neighbors?!")
        tree = cKDTree(bal.points)
        for i in rng.choice(len(idx), size=min(n, len(idx)), replace=False):
            _, near = tree.query(bal.points[idx[i]], k=min(11, len(bal.points)))
            idx[i] = int(rng.choice(np.atleast_1d(near)[1:]))      # .skip(1).take(10)
    return _with_graph(bal, g.offsets, idx, g.uv)
