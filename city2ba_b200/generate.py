"""Host mirror of city2ba::generate for the hot path (reference: src/generate.rs).

`Scene` stands where `embree_rs::CommittedScene` stood (src/bin/city2ba.rs:515-521) and
`visibility_graph` keeps the reference's signature and result order
(src/generate.rs:424-481); the work happens in libcity2ba_cuda.so.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import CAM_STRIDE, Obs, VisOptions, check, context, lib


def _cam_array(cameras) -> np.ndarray:
    """Accept an (C,15) array or a sequence of SnavelyCamera."""
    if isinstance(cameras, np.ndarray):
        a = np.ascontiguousarray(cameras, dtype=np.float64)
    elif len(cameras) and hasattr(cameras[0], "to_record"):
        a = np.stack([c.to_record() for c in cameras]) if len(cameras) else np.zeros((0, CAM_STRIDE))
    else:
        a = np.ascontiguousarray(cameras, dtype=np.float64)
    return a.reshape(-1, CAM_STRIDE)


def _pts_array(points) -> np.ndarray:
    return np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)


class Scene:
    """Triangle scene committed to a GPU LBVH (replaces Scene::new + model_to_geometry + commit)."""

    def __init__(self, xyz, tri, ctx: _lib.Context | None = None):
        self.ctx = ctx or context()
        xyz = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
        tri = np.ascontiguousarray(tri, dtype=np.uint32).reshape(-1, 3)
        self._h = C.c_void_p()
        check(lib().c2b_scene_create(
            self.ctx.handle, xyz.ctypes.data_as(C.POINTER(C.c_float)), xyz.shape[0],
            tri.ctypes.data_as(C.POINTER(C.c_uint32)), tri.shape[0], C.byref(self._h)))

    @classmethod
    def from_models(cls, models, ctx=None):
        """models: iterable of (positions f32 (nv,3), indices u32 (nt,3)) per OBJ object —
        the loop over `model_to_geometry` + `attach_geometry` (src/bin/city2ba.rs:517-520)."""
        xyz, tri, base = [], [], 0
        for pos, idx in models:
            pos = np.asarray(pos, dtype=np.float32).reshape(-1, 3)
            idx = np.asarray(idx, dtype=np.uint32).reshape(-1, 3)
            xyz.append(pos)
            tri.append(idx + np.uint32(base))
            base += pos.shape[0]
        if not xyz:
            return cls(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint32), ctx)
        return cls(np.concatenate(xyz), np.concatenate(tri), ctx)

    @property
    def handle(self):
        return self._h

    @property
    def num_triangles(self) -> int:
        return int(lib().c2b_scene_num_triangles(self._h))

    @property
    def num_nodes(self) -> int:
        return int(lib().c2b_scene_num_nodes(self._h))

    def bounds(self):
        """(lower xyz, upper xyz) as f32 — CommittedScene::bounds(), src/generate.rs:237."""
        lo = np.zeros(3, np.float32)
        hi = np.zeros(3, np.float32)
        check(lib().c2b_scene_bounds(self._h, lo.ctypes.data_as(C.POINTER(C.c_float)),
                                     hi.ctypes.data_as(C.POINTER(C.c_float))))
        return lo, hi

    def occluded(self, org, dirs, tfar) -> np.ndarray:
        """Embree-shaped any-hit on explicit f32 rays: returns a bool array (True = occluded)."""
        org = np.ascontiguousarray(org, np.float32).reshape(-1, 3)
        dirs = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        tfar = np.ascontiguousarray(tfar, np.float32).reshape(-1)
        n = org.shape[0]
        rays = np.zeros(n, dtype=np.dtype([
            ("org", np.float32, 3), ("tnear", np.float32), ("dir", np.float32, 3),
            ("time", np.float32), ("tfar", np.float32), ("mask", np.uint32), ("id", np.uint32),
            ("flags", np.uint32)]))
        assert rays.dtype.itemsize == 48
        rays["org"], rays["dir"], rays["tfar"] = org, dirs, tfar
        check(lib().c2b_occluded(self.ctx.handle, self._h,
                                 rays.ctypes.data_as(C.POINTER(_lib.Ray48)), n))
        return np.isneginf(rays["tfar"])

    def intersect(self, org, dirs, tfar=np.inf):
        """Embree-shaped closest hit on explicit f32 rays: (hit bool array, distance array; inf = miss)."""
        org = np.ascontiguousarray(org, np.float32).reshape(-1, 3)
        dirs = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        n = org.shape[0]
        rays = np.zeros(n, dtype=np.dtype([
            ("org", np.float32, 3), ("tnear", np.float32), ("dir", np.float32, 3),
            ("time", np.float32), ("tfar", np.float32), ("mask", np.uint32), ("id", np.uint32),
            ("flags", np.uint32)]))
        rays["org"], rays["dir"] = org, dirs
        rays["tfar"] = np.broadcast_to(np.asarray(tfar, np.float32), (n,))
        check(lib().c2b_intersect(self.ctx.handle, self._h, rays.ctypes.data_as(C.POINTER(_lib.Ray48)), n))
        hit = rays["flags"] != 0
        return hit, np.where(hit, rays["tfar"], np.float32(np.inf))

    def intersect1(self, org, direction):
        """Closest hit of one ray: (hit, distance) — scene.intersect, src/generate.rs:253-262."""
        o = np.ascontiguousarray(org, np.float32)
        d = np.ascontiguousarray(direction, np.float32)
        hit, t = C.c_int(0), C.c_float(0)
        check(lib().c2b_intersect1(self.ctx.handle, self._h, o.ctypes.data_as(C.POINTER(C.c_float)),
                                   d.ctypes.data_as(C.POINTER(C.c_float)), C.byref(hit), C.byref(t)))
        return bool(hit.value), float(t.value)

    def close(self):
        if self._h:
            lib().c2b_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class VisGraph:
    """CSR visibility graph.  Behaves like the reference's Vec<Vec<(usize,(f64,f64))>>:
    len(g) == cameras, g[i] -> list of (point_index, (u, v)) in ascending point index."""

    def __init__(self, offsets, point_idx, uv, stats=None):
        self.offsets = np.asarray(offsets, dtype=np.uint64)
        self.point_idx = np.asarray(point_idx, dtype=np.uint64)
        self.uv = np.asarray(uv, dtype=np.float64).reshape(-1, 2)
        self.stats = stats or {}

    def __len__(self):
        return len(self.offsets) - 1

    def __getitem__(self, i):
        a, b = int(self.offsets[i]), int(self.offsets[i + 1])
        return [(int(p), (float(u), float(v)))
                for p, (u, v) in zip(self.point_idx[a:b], self.uv[a:b])]

    def __iter__(self):
        for i in range(len(self)):
            yield self[i]

    @property
    def num_observations(self) -> int:
        return int(self.offsets[-1])

    def counts(self):
        return np.diff(self.offsets.astype(np.int64))


def _options(cull_mode, occlusion, endpoint_guard_rel, count_traversal, block_length, block_inset, predicate="watertight"):
    o = VisOptions()
    lib().c2b_vis_options_default(C.byref(o))
    o.cull_mode = {"grid": _lib.CULL_GRID, "exhaustive": _lib.CULL_EXHAUSTIVE}[cull_mode]
    o.occlusion = {"mesh": _lib.OCC_MESH, "none": _lib.OCC_NONE, "analytic": _lib.OCC_ANALYTIC}[occlusion]
    o.endpoint_guard_rel = int(bool(endpoint_guard_rel))
    o.count_traversal = int(bool(count_traversal))
    o.block_length = float(block_length)
    o.block_inset = float(block_inset)
    o.predicate = {"watertight": _lib.PRED_WATERTIGHT, "mt": _lib.PRED_MT}[predicate]
    return o


def _stats(o: Obs) -> dict:
    return {k: getattr(o, k) for k, _ in Obs._fields_ if k not in ("offsets", "point_idx", "uv")}


def visibility_graph(scene, cameras, points, max_dist, verbose=False, *, cull_mode="grid",
                     occlusion="mesh", endpoint_guard_rel=False, count_traversal=False,
                     block_length=20.0, block_inset=1.0, predicate="watertight", ctx=None) -> VisGraph:
    """Compute the camera-point visibility graph (src/generate.rs:424-481).

    scene: Scene or None (only with occlusion != "mesh").  cameras: (C,15) records or
    SnavelyCamera list.  points: (P,3).  Returns a VisGraph (camera-major CSR).
    `verbose` is accepted for signature parity; there is no progress bar (the call is one
    kernel pipeline).  predicate = "mt" decides occlusion with the Moeller-Trumbore test of Embree's default
    intersector (what the reference's scene runs) instead of the watertight default.
    """
    ctx = ctx or (scene.ctx if scene is not None else context())
    cams, pts = _cam_array(cameras), _pts_array(points)
    opt = _options(cull_mode, occlusion, endpoint_guard_rel, count_traversal, block_length, block_inset, predicate)
    out = Obs()
    check(lib().c2b_visibility_graph(
        ctx.handle, scene.handle if scene is not None else None, cams.ctypes.data, cams.shape[0],
        pts.ctypes.data, pts.shape[0], float(max_dist), C.byref(opt), C.byref(out)))
    Cn, O = int(out.n_cameras), int(out.n_obs)
    offsets = np.ctypeslib.as_array(out.offsets, shape=(Cn + 1,)).copy()
    if O:
        idx = np.ctypeslib.as_array(out.point_idx, shape=(O,)).copy()
        uv = np.ctypeslib.as_array(out.uv, shape=(2 * O,)).copy()
    else:
        idx, uv = np.zeros(0, np.uint32), np.zeros(0, np.float64)
    st = _stats(out)
    lib().c2b_obs_free(ctx.handle, C.byref(out))
    return VisGraph(offsets, idx, uv, st)


class MultiScene:
    """The triangle scene replicated on every GPU of a MultiContext (c2b_scene_create_multi)."""

    def __init__(self, xyz, tri, mctx: _lib.MultiContext):
        self.mctx = mctx
        xyz = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
        tri = np.ascontiguousarray(tri, dtype=np.uint32).reshape(-1, 3)
        self._h = C.c_void_p()
        check(lib().c2b_scene_create_multi(
            mctx.handle, xyz.ctypes.data_as(C.POINTER(C.c_float)), xyz.shape[0],
            tri.ctypes.data_as(C.POINTER(C.c_uint32)), tri.shape[0], C.byref(self._h)))

    @property
    def handle(self):
        return self._h

    def close(self):
        if self._h:
            lib().c2b_scene_destroy_multi(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def visibility_graph_multi(mctx, scene, cameras, points, max_dist, *, cull_mode="grid", occlusion="mesh",
                           endpoint_guard_rel=False, block_length=20.0, block_inset=1.0) -> VisGraph:
    """visibility_graph over the GPUs of `mctx` (camera ranges; c2b_visibility_graph_multi): ONE host CSR,
    identical to the single-GPU result.  stats["multi"] holds the per-GPU ranges, counts and stage times."""
    cams, pts = _cam_array(cameras), _pts_array(points)
    opt = _options(cull_mode, occlusion, endpoint_guard_rel, False, block_length, block_inset)
    out, ms = Obs(), _lib.MultiStats()
    check(lib().c2b_visibility_graph_multi(
        mctx.handle, scene.handle if scene is not None else None, cams.ctypes.data, cams.shape[0],
        pts.ctypes.data, pts.shape[0], float(max_dist), C.byref(opt), C.byref(out), C.byref(ms)))
    Cn, O = int(out.n_cameras), int(out.n_obs)
    offsets = np.ctypeslib.as_array(out.offsets, shape=(Cn + 1,)).copy()
    idx = np.ctypeslib.as_array(out.point_idx, shape=(O,)).copy() if O else np.zeros(0, np.uint32)
    uv = np.ctypeslib.as_array(out.uv, shape=(2 * O,)).copy() if O else np.zeros(0)
    st = _stats(out)
    G = ms.n_gpus
    st["multi"] = {k: [getattr(ms, k)[g] for g in range(G)] for k in
                   ("cam_begin", "cam_end", "n_obs", "obs_base", "ms_points", "ms_compute", "ms_exchange", "ms_d2h")}
    st["multi"]["ms_wall"] = ms.ms_wall
    return VisGraph(offsets, idx, uv, st)


class ResidentProblem:
    """Keeps cameras / points / result in HBM between calls (the three-call form of the ABI)."""

    def __init__(self, ctx=None):
        self.ctx = ctx or context()

    def upload_points(self, points):
        p = _pts_array(points)
        check(lib().c2b_upload_points(self.ctx.handle, p.ctypes.data, p.shape[0]))

    def upload_cameras(self, cameras):
        c = _cam_array(cameras)
        check(lib().c2b_upload_cameras(self.ctx.handle, c.ctypes.data, c.shape[0]))

    def upload_points_ptr(self, ptr: int, n: int):
        check(lib().c2b_upload_points(self.ctx.handle, ptr, n))

    def upload_cameras_ptr(self, ptr: int, n: int):
        check(lib().c2b_upload_cameras(self.ctx.handle, ptr, n))

    def run(self, scene, max_dist, **kw) -> dict:
        opt = _options(kw.get("cull_mode", "grid"), kw.get("occlusion", "mesh"),
                       kw.get("endpoint_guard_rel", False), kw.get("count_traversal", False),
                       kw.get("block_length", 20.0), kw.get("block_inset", 1.0))
        out = Obs()
        check(lib().c2b_visibility_graph_resident(
            self.ctx.handle, scene.handle if scene is not None else None, float(max_dist),
            C.byref(opt), C.byref(out)))
        return _stats(out)

    def download(self) -> VisGraph:
        out = Obs()
        check(lib().c2b_download_obs(self.ctx.handle, C.byref(out)))
        Cn, O = int(out.n_cameras), int(out.n_obs)
        offsets = np.ctypeslib.as_array(out.offsets, shape=(Cn + 1,)).copy()
        idx = np.ctypeslib.as_array(out.point_idx, shape=(O,)).copy() if O else np.zeros(0, np.uint32)
        uv = np.ctypeslib.as_array(out.uv, shape=(2 * O,)).copy() if O else np.zeros(0)
        return VisGraph(offsets, idx, uv, _stats(out))

    def download_raw(self) -> Obs:
        """Download into the ctx's pinned buffers without copying to numpy (bench e2e)."""
        out = Obs()
        check(lib().c2b_download_obs(self.ctx.handle, C.byref(out)))
        return out

    # ---- the noise pass on the resident problem (no PCIe traffic) ----
    def add_drift(self, strength, angle_strength, std, direction=None, seed=0):
        """noise::add_drift on the resident cameras / points; direction None = add_drift_normalized"""
        d = None if direction is None else np.ascontiguousarray(direction, np.float64).ctypes.data_as(C.POINTER(C.c_double))
        check(lib().c2b_add_drift_resident(self.ctx.handle, float(strength), float(angle_strength), float(std), d, int(seed)))

    def add_noise(self, translation_std, rotation_std, point_std, observations_std, seed=0):
        check(lib().c2b_add_noise_resident(self.ctx.handle, float(translation_std), float(rotation_std),
                                           float(point_std), float(observations_std), int(seed)))

    def add_sin_noise(self, direction, noise_direction, strength, frequency):
        """noise::add_sin_noise on the resident cameras / points (dimensions from their extent)"""
        pd = C.POINTER(C.c_double)
        d = np.ascontiguousarray(direction, np.float64)
        nd = np.ascontiguousarray(noise_direction, np.float64)
        check(lib().c2b_add_sin_noise_resident(self.ctx.handle, d.ctypes.data_as(pd), nd.ctypes.data_as(pd),
                                               float(strength), float(frequency)))

    def download_problem(self, num_cameras: int, num_points: int):
        cams, pts = np.empty((num_cameras, CAM_STRIDE)), np.empty((num_points, 3))
        pd = C.POINTER(C.c_double)
        check(lib().c2b_download_problem(self.ctx.handle, cams.ctypes.data_as(pd), pts.ctypes.data_as(pd)))
        return cams, pts

    def reprojection_error(self, norm: float) -> float:
        v = C.c_double(0)
        check(lib().c2b_reprojection_error_resident(self.ctx.handle, float(norm), C.byref(v)))
        return v.value

    def cull(self) -> dict:
        """BAProblem::cull (LCC + remove_singletons to a fixed point) on the resident problem, in HBM.  Afterwards
        download / download_problem / reprojection_error / add_* and a new run see the culled problem.  Returns
        the stats: n_cameras, n_points, n_obs after the cull, iterations, ms_compute (device time)."""
        st = _lib.CullStats()
        check(lib().c2b_cull_problem_resident(self.ctx.handle, C.byref(st)))
        return st.to_dict()

    def add_incorrect_correspondences(self, mismatch_chance, seed=0) -> dict:
        """noise::add_incorrect_correspondences on the resident CSR, in HBM (c2b_add_incorrect_correspondences_resident):
        the draws of noise.add_incorrect_correspondences_gpu.  Afterwards download / reprojection_error / cull / write
        see the edited graph.  Raises AssertionError (AllWeightsZero / NegativeWeight) and leaves the problem unchanged
        when a selected observation's weights are invalid.  Returns the stats: n_selected, n_swapped, ms_compute."""
        from .noise import _weight_error
        st = _lib.MismatchStats()
        try:
            check(lib().c2b_add_incorrect_correspondences_resident(self.ctx.handle, float(mismatch_chance),
                                                                   int(seed) & (2 ** 64 - 1), C.byref(st)))
        except _lib.C2BError as e:
            a = _weight_error(e)
            if a is not None:
                raise a from e
            raise
        return st.to_dict()

    def write(self, path) -> dict:
        """BAProblem::write of the resident problem (c2b_write_bal_resident): .bal text or .bbal binary by the
        extension, encoded on the GPU and streamed to disk.  Returns the stats: bytes, chunks, ms_encode, ms_d2h
        (device time), ms_write (host time in write(2))."""
        from .baproblem import BAProblem, IOError_
        fmt = _lib.BAL_BINARY if BAProblem._bal_binary(path) else _lib.BAL_TEXT
        st = _lib.BalStats()
        try:
            check(lib().c2b_write_bal_resident(self.ctx.handle, str(path).encode(), fmt, C.byref(st)))
        except _lib.C2BError as e:
            if e.code == _lib.ERR_IO:
                raise IOError_(str(e)) from e
            raise
        return st.to_dict()

    def read(self, path) -> dict:
        """BAProblem::from_file into HBM (c2b_read_bal_resident): .bal text or .bbal binary by the extension, streamed
        to the device and parsed there.  The file's problem replaces the resident one; afterwards download /
        download_problem / reprojection_error / add_* / cull / write see it.  Raises ParseError on a malformed or
        short file, IOError_ when it cannot be read, AssertionError on an observation index out of range (the errors
        of BAProblem.from_file).  Returns the stats: n_cameras, n_points, n_obs, bytes, chunks, slow_tokens (numbers
        converted on the host), regrouped, ms_read (host time in pread(2)), ms_h2d, ms_parse (device time)."""
        from .baproblem import BAProblem, IOError_, ParseError
        fmt = _lib.BAL_BINARY if BAProblem._bal_binary(path) else _lib.BAL_TEXT
        st = _lib.BalReadStats()
        try:
            check(lib().c2b_read_bal_resident(self.ctx.handle, str(path).encode(), fmt, C.byref(st)))
        except _lib.C2BError as e:
            if e.code == _lib.ERR_PARSE:
                raise ParseError(str(e)) from e
            if e.code == _lib.ERR_IO:
                raise IOError_(str(e)) from e
            if e.code == _lib.ERR_INVALID and "index out of range" in str(e):
                raise AssertionError(str(e)) from e
            raise
        return st.to_dict()


def generate_world_points_uniform(xyz, tri, cameras, num_points, max_dist, seed=None, ctx=None) -> np.ndarray:
    """src/generate.rs:356-420 on the GPU: `num_points` points on the mesh (area-weighted triangle,
    uniform inside it) that lie within `max_dist` of some camera.  `xyz`/`tri` are all models'
    vertices / index triples concatenated.  The reference draws from thread_rng(); here the sample is a
    pure function of `seed` (default: a fresh one from os.urandom)."""
    import os
    ctx = ctx or context()
    xyz = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
    tri = np.ascontiguousarray(tri, dtype=np.uint32).reshape(-1, 3)
    cams = _cam_array(cameras)
    seed = int.from_bytes(os.urandom(8), "little") if seed is None else int(seed) & (2 ** 64 - 1)
    out = np.empty((int(num_points), 3))
    n = C.c_uint64(0)
    check(lib().c2b_generate_world_points_uniform(
        ctx.handle, xyz.ctypes.data_as(C.POINTER(C.c_float)), xyz.shape[0],
        tri.ctypes.data_as(C.POINTER(C.c_uint32)), tri.shape[0], cams.ctypes.data_as(C.POINTER(C.c_double)),
        cams.shape[0], int(num_points), float(max_dist), seed, out.ctypes.data_as(C.POINTER(C.c_double)),
        C.byref(n)))
    return out[: n.value]


# ---- OBJ ingest and camera generators (src/generate.rs:109-280, 484-544; src/bin/city2ba.rs:481-538) -------
# Host side, like the reference's; the same procedures as include/city2ba.hpp (seeded where the reference
# draws from thread_rng(), so parity with it is distributional).

class Model:
    """tobj::Model: name + per-model vertex array (only the vertices its elements use, in order of first
    use) + flat index list (triangles; `l` records append index pairs)."""

    def __init__(self, name, positions, indices):
        self.name = name
        self.positions = np.asarray(positions, np.float32).reshape(-1, 3)
        self.indices = np.asarray(indices, np.uint32).reshape(-1)


def load_obj(path) -> list:
    """tobj 0.1.12's rules (src/bin/city2ba.rs:481): one Model per `o` / `g` that is followed by elements;
    quads as (a,b,c),(a,c,d), larger polygons as a fan from their first vertex; `l` records keep two indices,
    `p` records one; materials are not read."""
    from .baproblem import IOError_
    try:
        fh = open(path)
    except OSError as e:
        raise IOError_(f'Could not open file "{path}"') from e
    pos, n_vt, n_vn = [], 0, 0
    models, faces, name = [], [], "unnamed_object"

    def flush():
        nonlocal faces
        if not faces:
            return
        seen, positions, indices = {}, [], []

        def add(k):
            if k not in seen:
                seen[k] = len(positions)
                positions.append(pos[k[0]])
            indices.append(seen[k])
        for e in faces:
            if len(e) <= 3:
                order = range(len(e))
            elif len(e) == 4:
                order = (0, 1, 2, 0, 2, 3)
            else:
                order = [j for i in range(1, len(e) - 1) for j in (0, i, i + 1)]
            for i in order:
                add(e[i])
        models.append(Model(name, positions, indices))
        faces = []

    with fh:
        for lineno, line in enumerate(fh, 1):
            t = line.split()
            if not t or t[0].startswith("#"):
                continue
            if t[0] == "v":
                pos.append(tuple(float(x) for x in t[1:4]))
            elif t[0] == "vt":
                n_vt += 1
            elif t[0] == "vn":
                n_vn += 1
            elif t[0] in ("f", "l", "p"):
                e = []
                for tok in t[1:]:
                    parts = (tok.split("/") + ["", ""])[:3]
                    key = []
                    for part, n in zip(parts, (len(pos), n_vt, n_vn)):
                        i = int(part) if part else 0
                        key.append(i - 1 if i > 0 else n + i if i < 0 else -1)
                    if not 0 <= key[0] < len(pos):
                        raise IOError_(f"Load error: face vertex index out of range ({path}:{lineno})")
                    e.append(tuple(key))
                if not e:
                    raise IOError_(f"Load error: face parse error ({path}:{lineno})")
                faces.append(e)
            elif t[0] in ("o", "g"):
                flush()
                name = line.split(None, 1)[1].strip() if len(t) > 1 else "unnamed_object"
    flush()
    return models


def concat_models(models):
    """all models as one (xyz, tri) pair for Scene / the point sampler: each model's index list regrouped
    into triples on its own (num_tri = indices.len() / 3, src/generate.rs:78) and offset"""
    xyz, tri, base = [], [], 0
    for m in models:
        xyz.append(m.positions)
        n = len(m.indices) // 3 * 3
        tri.append(m.indices[:n].reshape(-1, 3) + np.uint32(base))
        base += len(m.positions)
    if not xyz:
        return np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint32)
    return np.concatenate(xyz), np.concatenate(tri).astype(np.uint32)


def move_to_origin(models):
    """src/generate.rs:484-527"""
    mn = np.min([m.positions.min(axis=0) for m in models if len(m.positions)], axis=0)
    return [Model(m.name, m.positions - mn, m.indices) for m in models]


def modify_intrinsics(cameras, intrinsic_start, intrinsic_end, seed=None):
    """src/generate.rs:530-544: intrinsics uniform in [start, end); returns a new (C,15) array"""
    cams = _cam_array(cameras).copy()
    rng = np.random.default_rng(seed)
    s, e = np.asarray(intrinsic_start, float), np.asarray(intrinsic_end, float)
    cams[:, 12:15] = s + rng.uniform(size=(len(cams), 3)) * (e - s)
    return cams


def _path_segments(path: Model):
    v = path.positions.astype(np.float64)
    idx = path.indices[: len(path.indices) // 2 * 2].reshape(-1, 2)
    return v[idx[:, 0]], v[idx[:, 1]]


def _camera_looking_along(pos, direction):
    from .baproblem import SnavelyCamera, between_vectors
    d = direction / np.linalg.norm(direction)
    return SnavelyCamera.from_position_direction(pos, between_vectors(d, np.array([0.0, 0.0, -1.0]))).to_record()


def generate_cameras_path(scene, path: Model, num_cameras, seed=None):
    """src/generate.rs:109-148: random positions along the path (segments weighted by length), looking along it"""
    a, b = _path_segments(path)
    length = np.linalg.norm(b - a, axis=1)
    if not length.sum() > 0:
        raise AssertionError("called `Result::unwrap()` on an `Err` value: AllWeightsZero")
    rng = np.random.default_rng(seed)
    cams = np.empty((num_cameras, CAM_STRIDE))
    for k, i in enumerate(rng.choice(len(a), size=num_cameras, p=length / length.sum())):
        cams[k] = _camera_looking_along(a[i] + rng.uniform() * (b[i] - a[i]), b[i] - a[i])
    return cams


def generate_cameras_path_step(scene, path: Model, num_cameras, step_size):
    """src/generate.rs:152-213: fixed steps from the start of the path"""
    a, b = _path_segments(path)
    length = np.linalg.norm(b - a, axis=1)
    total = float(length.sum())
    assert num_cameras * step_size <= total, (
        f"Length of path {total} is less than the number of cameras ({num_cameras}) times the step size "
        f"({step_size}) {num_cameras * step_size}")
    seg, dist = 0, 0.0
    cams = np.empty((num_cameras, CAM_STRIDE))
    for k in range(num_cameras):
        d = b[seg] - a[seg]                       # IndexError = the reference's out-of-bounds panic
        cams[k] = _camera_looking_along(a[seg] + dist / length[seg] * d, d)
        dist += step_size
        while dist >= length[seg]:
            dist -= length[seg]
            seg += 1
            length[seg]                           # the reference indexes the next segment here
    return cams


def _poisson_disk(samples, rng):
    """Bridson dart throwing in the unit square at the hexagonal-packing radius for `samples` discs (the
    reference's `poisson` crate, Ebeida's sampler at relative radius 1, is not vendored)"""
    if samples == 0:
        return np.zeros((0, 2))
    r = 2.0 * np.sqrt(0.9068996821171089 / (samples * np.pi))
    cell = r / np.sqrt(2.0)
    n = max(1, int(np.ceil(1.0 / cell)))
    grid = -np.ones((n, n), np.int64)
    out, active = [], []

    def cell_of(x):
        return min(n - 1, int(x / cell))

    def fits(x, y):
        cx, cy = cell_of(x), cell_of(y)
        for j in range(max(0, cy - 2), min(n - 1, cy + 2) + 1):
            for i in range(max(0, cx - 2), min(n - 1, cx + 2) + 1):
                k = grid[j, i]
                if k >= 0 and (out[k][0] - x) ** 2 + (out[k][1] - y) ** 2 < r * r:
                    return False
        return True

    def push(x, y):
        grid[cell_of(y), cell_of(x)] = len(out)
        active.append(len(out))
        out.append((x, y))

    push(rng.uniform(), rng.uniform())
    while active:
        a = int(rng.integers(len(active)))
        bx, by = out[active[a]]
        for _ in range(30):
            ang, rad = rng.uniform(0.0, 2.0 * np.pi), r * np.sqrt(rng.uniform(1.0, 4.0))
            x, y = bx + rad * np.cos(ang), by + rad * np.sin(ang)
            if 0.0 <= x < 1.0 and 0.0 <= y < 1.0 and fits(x, y):
                push(x, y)
                break
        else:
            active[a] = active[-1]
            active.pop()
    return np.array(out)


def generate_cameras_poisson(scene: Scene, num_points, height, ground, seed=None):
    """src/generate.rs:217-280: Poisson-disk positions over the scene's (x, z) bounds, dropped onto the tallest
    surface below them (ALL downward closest-hit rays in one GPU batch), raised by `height`, kept if
    pt[2] < lower_y + ground (z against y, as the reference writes it, :264), random yaw about y"""
    from .baproblem import SnavelyCamera, from_angle_y
    rng = np.random.default_rng(seed)
    smp = _poisson_disk(num_points * 2, rng)
    lo, hi = scene.bounds()
    start = np.array([float(hi[0]), float(hi[1]) + 0.1, float(hi[2])])
    delta = np.array([float(hi[0] - lo[0]), 0.0, float(hi[2] - lo[2])])
    origins = start - delta * np.stack([smp[:, 0], np.zeros(len(smp)), smp[:, 1]], axis=1)
    if not len(origins):
        return np.zeros((0, CAM_STRIDE))
    hit, t = scene.intersect(origins, np.tile(np.array([0.0, -1.0, 0.0], np.float32), (len(origins), 1)))
    cams = []
    for o, h, tt in zip(origins, hit, t):
        if not h:
            continue
        pt = o + np.array([0.0, -1.0, 0.0]) * float(tt) + np.array([0.0, height, 0.0])
        if pt[2] < float(lo[1]) + ground:
            cams.append(SnavelyCamera.from_position_direction(pt, from_angle_y(rng.uniform(0.0, 2.0 * np.pi))).to_record())
    return np.array(cams).reshape(-1, CAM_STRIDE)
