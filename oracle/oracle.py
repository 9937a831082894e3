"""ctypes binding of the CPU ORACLE (oracle/liboracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package (city2ba_b200/) never imports it.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liboracle.so")

CAM = 15


def build(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, f) for f in ("cpu_ref.c", "c2b_oracle.c", "c2b_oracle.h")]
    if force or not os.path.exists(_SO) or any(
        os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs
    ):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _SO


class _Vis(C.Structure):
    _fields_ = [
        ("n_cameras", C.c_uint64),
        ("n_candidates", C.c_uint64),
        ("n_obs", C.c_uint64),
        ("cand_offsets", C.POINTER(C.c_uint64)),
        ("cand_point", C.POINTER(C.c_uint64)),
        ("cand_uv", C.POINTER(C.c_double)),
        ("cand_occluded", C.POINTER(C.c_uint8)),
        ("cand_flags", C.POINTER(C.c_uint8)),
        ("offsets", C.POINTER(C.c_uint64)),
        ("point_idx", C.POINTER(C.c_uint64)),
        ("uv", C.POINTER(C.c_double)),
        ("n_flag_edge", C.c_uint64),
        ("n_flag_graze", C.c_uint64),
        ("n_flag_endpoint", C.c_uint64),
        ("n_flag_cull", C.c_uint64),
    ]


_lib = None


def build_native(out_dir: str) -> str:
    """-O3 -march=native build of the same sources for the TIMED CPU arm, made by the process that runs it (a
    build made on another CPU may not run here) into `out_dir`, outside the checkout, which may be read-only."""
    so = os.path.join(out_dir, "liboracle_native.so")
    subprocess.check_call(["make", "-C", _HERE, "-s", "native", f"NATIVE_OUT={so}"])
    return so


def lib():
    """C2B_ORACLE_NATIVE=1 (set by bench.py for its CPU arms) selects the -march=native build."""
    global _lib
    if _lib is None:
        if os.environ.get("C2B_ORACLE_NATIVE") == "1":
            with tempfile.TemporaryDirectory(prefix="c2b_oracle_native_") as d:
                _lib = C.CDLL(build_native(d))   # stays mapped after the directory is removed
        else:
            build()
            _lib = C.CDLL(_SO)
        _lib.orc_visibility_graph.restype = C.POINTER(_Vis)
        _lib.orc_ref_visibility_graph.restype = C.POINTER(_Vis)
        _lib.orc_synthetic_visibility.restype = C.POINTER(_Vis)
        _lib.orc_grid_num_cameras.restype = C.c_uint64
        _lib.orc_grid_num_points.restype = C.c_uint64
        _lib.orc_deg_to_rad.restype = C.c_double
        _lib.orc_deg_to_rad.argtypes = [C.c_double]
        _lib.orc_total_reprojection_error.restype = C.c_double
        _lib.orc_hits_building.restype = C.c_int
        _lib.orc_ray_triangle.restype = C.c_int
    return _lib


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a, t=C.c_double):
    return a.ctypes.data_as(C.POINTER(t))


def _u64(x):
    return C.c_uint64(int(x))


# ---- camera math -------------------------------------------------------------------------
def _call3(fn, cam, p, n_out):
    cam, p = _d(cam), _d(p)
    out = np.empty(n_out)
    getattr(lib(), fn)(_p(cam), _p(p), _p(out))
    return out


def project_world(cam, p):
    return _call3("orc_project_world", cam, p, 3)


def project(cam, pc):
    return _call3("orc_project", cam, pc, 2)


def to_world(cam, p):
    return _call3("orc_to_world", cam, p, 3)


def center(cam):
    cam = _d(cam)
    out = np.empty(3)
    lib().orc_center(_p(cam), _p(out))
    return out


def from_position_direction(pos, R):
    pos, R = _d(pos), _d(R)
    out = np.empty(CAM)
    lib().orc_from_position_direction(_p(pos), _p(R), _p(out))
    return out


def transform(cam, dR, dloc):
    cam, dR, dloc = _d(cam), _d(dR), _d(dloc)
    out = np.empty(CAM)
    lib().orc_transform(_p(cam), _p(dR), _p(dloc), _p(out))
    return out


def from_rodrigues(v):
    v = _d(v)
    out = np.empty(9)
    lib().orc_from_rodrigues(_p(v), _p(out))
    return out


def to_rodrigues(R):
    R = _d(R)
    out = np.empty(3)
    lib().orc_to_rodrigues(_p(R), _p(out))
    return out


def from_vec(v9):
    v9 = _d(v9)
    out = np.empty(CAM)
    lib().orc_from_vec(_p(v9), _p(out))
    return out


def to_vec(cam):
    cam = _d(cam)
    out = np.empty(9)
    lib().orc_to_vec(_p(cam), _p(out))
    return out


def from_angle_y(rad):
    out = np.empty(9)
    lib().orc_from_angle_y(C.c_double(rad), _p(out))
    return out


def from_angle_x(rad):
    out = np.empty(9)
    lib().orc_from_angle_x(C.c_double(rad), _p(out))
    return out


def from_axis_angle(axis, rad):
    axis = _d(axis)
    out = np.empty(9)
    lib().orc_from_axis_angle(_p(axis), C.c_double(rad), _p(out))
    return out


def deg_to_rad(deg):
    return lib().orc_deg_to_rad(float(deg))


# ---- visibility --------------------------------------------------------------------------
class Vis:
    """numpy copy of an orc_vis result."""

    def __init__(self, ptr, with_cands=True):
        v = ptr.contents
        Cn, nc, no = int(v.n_cameras), int(v.n_candidates), int(v.n_obs)
        self.n_cameras, self.n_candidates, self.n_obs = Cn, nc, no

        def arr(p, n, dt):
            if not p or n == 0:
                return np.zeros(0, dtype=dt)
            return np.ctypeslib.as_array(p, shape=(n,)).astype(dt, copy=True)

        self.offsets = arr(v.offsets, Cn + 1, np.uint64)
        self.point_idx = arr(v.point_idx, no, np.uint64)
        self.uv = arr(v.uv, 2 * no, np.float64).reshape(-1, 2)
        if with_cands and v.cand_offsets:
            self.cand_offsets = arr(v.cand_offsets, Cn + 1, np.uint64)
            self.cand_point = arr(v.cand_point, nc, np.uint64)
            self.cand_uv = arr(v.cand_uv, 2 * nc, np.float64).reshape(-1, 2)
            self.cand_occluded = arr(v.cand_occluded, nc, np.uint8)
            self.cand_flags = arr(v.cand_flags, nc, np.uint8)
        self.n_flag_edge = int(v.n_flag_edge)
        self.n_flag_graze = int(v.n_flag_graze)
        self.n_flag_endpoint = int(v.n_flag_endpoint)
        self.n_flag_cull = int(v.n_flag_cull)
        lib().orc_vis_free(ptr)


def _mesh(xyz, tri):
    xyz = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1)
    tri = np.ascontiguousarray(tri, dtype=np.uint32).reshape(-1)
    return xyz, tri


def visibility_graph(xyz, tri, cams, pts, max_dist, endpoint_guard_rel=False, want_flags=False):
    xyz, tri = _mesh(xyz, tri)
    cams, pts = _d(cams).reshape(-1), _d(pts).reshape(-1)
    r = lib().orc_visibility_graph(
        _p(xyz, C.c_float), _u64(xyz.size // 3), _p(tri, C.c_uint32), _u64(tri.size // 3),
        _p(cams), _u64(cams.size // CAM), _p(pts), _u64(pts.size // 3), C.c_double(max_dist),
        C.c_int(int(endpoint_guard_rel)), C.c_int(int(want_flags)))
    return Vis(r)


def occluded_mt(xyz, tri, cams, pts, vis, endpoint_guard_rel=False):
    """occluded verdict of every candidate of `vis` under the restatement of Embree's default
    Moeller-Trumbore intersector (A/B counter against the watertight predicate; unpinned)."""
    xyz, tri = _mesh(xyz, tri)
    cams, pts = _d(cams).reshape(-1), _d(pts).reshape(-1)
    off = np.ascontiguousarray(vis.cand_offsets, dtype=np.uint64)
    cp = np.ascontiguousarray(vis.cand_point, dtype=np.uint64)
    out = np.zeros(len(cp), dtype=np.uint8)
    lib().orc_occluded_mt(
        _p(xyz, C.c_float), _u64(xyz.size // 3), _p(tri, C.c_uint32), _u64(tri.size // 3), _p(cams),
        _u64(cams.size // CAM), _p(pts), _p(off, C.c_uint64), _p(cp, C.c_uint64), C.c_int(int(endpoint_guard_rel)),
        _p(out, C.c_uint8))
    return out


def ref_visibility_graph(xyz, tri, cams, pts, max_dist, endpoint_guard_rel=False, n_threads=0):
    """Multithreaded CPU arm (OpenMP over cameras + CPU BVH).  Returns (Vis, threads_used)."""
    xyz, tri = _mesh(xyz, tri)
    cams, pts = _d(cams).reshape(-1), _d(pts).reshape(-1)
    used = C.c_int(0)
    r = lib().orc_ref_visibility_graph(
        _p(xyz, C.c_float), _u64(xyz.size // 3), _p(tri, C.c_uint32), _u64(tri.size // 3),
        _p(cams), _u64(cams.size // CAM), _p(pts), _u64(pts.size // 3), C.c_double(max_dist),
        C.c_int(int(endpoint_guard_rel)), C.c_int(int(n_threads)), C.byref(used))
    return Vis(r, with_cands=False), used.value


def synthetic_visibility(cams, pts, max_dist, analytic, block_length=20.0, block_inset=1.0):
    cams, pts = _d(cams).reshape(-1), _d(pts).reshape(-1)
    r = lib().orc_synthetic_visibility(
        _p(cams), _u64(cams.size // CAM), _p(pts), _u64(pts.size // 3), C.c_double(max_dist),
        C.c_int(int(analytic)), C.c_double(block_length), C.c_double(block_inset))
    return Vis(r)


def make_ray(center3, point3):
    c, p = _d(center3), _d(point3)
    out = np.empty(7, dtype=np.float32)
    lib().orc_make_ray(_p(c), _p(p), _p(out, C.c_float))
    return out  # org[3], dir[3], tfar


def ray_triangle(ray7, v0, v1, v2):
    r = np.ascontiguousarray(ray7, dtype=np.float32)
    a, b, c = (np.ascontiguousarray(v, dtype=np.float32) for v in (v0, v1, v2))
    return int(lib().orc_ray_triangle(_p(r, C.c_float), _p(a, C.c_float), _p(b, C.c_float),
                                      _p(c, C.c_float)))


def hits_building(c3, p3, block_length, block_inset):
    c, p = _d(c3), _d(p3)
    return int(lib().orc_hits_building(_p(c), _p(p), C.c_double(block_length),
                                       C.c_double(block_inset)))


# ---- synthetic inputs --------------------------------------------------------------------
def grid_cameras(cpb, n_blocks, block_length=20.0, camera_height=1.0):
    n = int(lib().orc_grid_num_cameras(_u64(cpb), _u64(n_blocks)))
    out = np.empty((n, CAM))
    lib().orc_grid_cameras(_u64(cpb), _u64(n_blocks), C.c_double(block_length),
                           C.c_double(camera_height), _p(out))
    return out


def grid_points(ppb, n_blocks, block_length=20.0, block_inset=1.0, point_height=1.0):
    n = int(lib().orc_grid_num_points(_u64(ppb), _u64(n_blocks)))
    out = np.empty((n, 3))
    lib().orc_grid_points(_u64(ppb), _u64(n_blocks), C.c_double(block_length),
                          C.c_double(block_inset), C.c_double(point_height), _p(out))
    return out


def line_cameras(num_cameras, length, camera_height):
    out = np.empty((num_cameras, CAM))
    lib().orc_line_cameras(_u64(num_cameras), C.c_double(length), C.c_double(camera_height), _p(out))
    return out


def line_points(num_points, length, point_offset, point_height):
    out = np.empty((num_points, 3))
    lib().orc_line_points(_u64(num_points), C.c_double(length), C.c_double(point_offset),
                          C.c_double(point_height), _p(out))
    return out


def city_mesh(n_blocks, block_length=20.0, block_inset=1.0, height=10.0):
    nb = n_blocks * n_blocks
    xyz = np.empty((8 * nb, 3), dtype=np.float32)
    tri = np.empty((12 * nb, 3), dtype=np.uint32)
    lib().orc_city_mesh(_u64(n_blocks), C.c_double(block_length), C.c_double(block_inset),
                        C.c_double(height), _p(xyz, C.c_float), _p(tri, C.c_uint32))
    return xyz, tri


# ---- noise -------------------------------------------------------------------------------
def philox4x32_10(ctr, key):
    ctr = np.ascontiguousarray(ctr, dtype=np.uint32)
    key = np.ascontiguousarray(key, dtype=np.uint32)
    out = np.empty(4, dtype=np.uint32)
    lib().orc_philox4x32_10(_p(ctr, C.c_uint32), _p(key, C.c_uint32), _p(out, C.c_uint32))
    return out


def unit2(w):
    """(cos, sin)(2 pi w / 2^32) as the noise draws evaluate it"""
    c, s = C.c_double(0), C.c_double(0)
    lib().orc_unit2(C.c_uint32(int(w)), C.byref(c), C.byref(s))
    return c.value, s.value


def neg2ln40(n40):
    f = lib().orc_neg2ln40
    f.restype = C.c_double
    return f(_u64(n40))


def normal40(a, b):
    f = lib().orc_normal40
    f.restype = C.c_double
    return f(C.c_uint32(int(a)), C.c_uint32(int(b)))


def sphere(a, b):
    out = np.empty(3)
    lib().orc_sphere(C.c_uint32(int(a)), C.c_uint32(int(b)), _p(out))
    return out


def noise_draws(words):
    """vectorised helper for the distribution tests: words (n, 4) uint32 -> dict of the draws one Philox
    block supplies: circle from word 0, sphere from words 0-1, N(0,1) from words 2-3"""
    w = np.ascontiguousarray(words, dtype=np.uint32).reshape(-1, 4)
    n = len(w)
    circle, sph, nrm = np.empty((n, 2)), np.empty((n, 3)), np.empty(n)
    f = lib().orc_noise_draws
    f(_p(w, C.c_uint32), _u64(n), _p(circle), _p(sph), _p(nrm))
    return {"circle": circle, "sphere": sph, "normal": nrm}


def mean(cams, pts):
    cams, pts = _d(cams).reshape(-1), _d(pts).reshape(-1)
    out = np.empty(3)
    lib().orc_mean(_p(cams), _u64(cams.size // CAM), _p(pts), _u64(pts.size // 3), _p(out))
    return out


def std(cams, pts):
    cams, pts = _d(cams).reshape(-1), _d(pts).reshape(-1)
    out = np.empty(3)
    lib().orc_std(_p(cams), _u64(cams.size // CAM), _p(pts), _u64(pts.size // 3), _p(out))
    return out


def add_drift(cams, pts, strength, angle_strength, std_, direction, seed):
    cams, pts = _d(cams).copy().reshape(-1, CAM), _d(pts).copy().reshape(-1, 3)
    d = _d(direction)
    lib().orc_add_drift(_p(cams), _u64(len(cams)), _p(pts), _u64(len(pts)), C.c_double(strength),
                        C.c_double(angle_strength), C.c_double(std_), _p(d), _u64(seed))
    return cams, pts


def add_drift_normalized(cams, pts, strength, angle_strength, std_, seed):
    cams, pts = _d(cams).copy().reshape(-1, CAM), _d(pts).copy().reshape(-1, 3)
    lib().orc_add_drift_normalized(_p(cams), _u64(len(cams)), _p(pts), _u64(len(pts)),
                                   C.c_double(strength), C.c_double(angle_strength),
                                   C.c_double(std_), _u64(seed))
    return cams, pts


def add_noise(cams, pts, uv, translation_std, rotation_std, point_std, observations_std, seed):
    cams, pts = _d(cams).copy().reshape(-1, CAM), _d(pts).copy().reshape(-1, 3)
    uv = _d(uv).copy().reshape(-1, 2)
    lib().orc_add_noise(_p(cams), _u64(len(cams)), _p(pts), _u64(len(pts)), _p(uv), _u64(len(uv)),
                        C.c_double(translation_std), C.c_double(rotation_std),
                        C.c_double(point_std), C.c_double(observations_std), _u64(seed))
    return cams, pts, uv


def generate_world_points_uniform(xyz, tri, cams, num_points, max_dist, seed):
    xyz = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
    tri = np.ascontiguousarray(tri, dtype=np.uint32).reshape(-1, 3)
    cams = _d(cams).reshape(-1, CAM)
    out = np.empty((int(num_points), 3))
    f = lib().orc_generate_world_points_uniform
    f.restype = C.c_uint64
    n = f(_p(xyz, C.c_float), _u64(len(xyz)), _p(tri, C.c_uint32), _u64(len(tri)), _p(cams), _u64(len(cams)),
          _u64(num_points), C.c_double(max_dist), _u64(seed), _p(out))
    return out[:int(n)]


def add_sin_noise(cams, pts, dir, noise_dir, strength, frequency):
    cams, pts = _d(cams).copy().reshape(-1, CAM), _d(pts).copy().reshape(-1, 3)
    lib().orc_add_sin_noise(_p(cams), _u64(len(cams)), _p(pts), _u64(len(pts)), _p(_d(dir)), _p(_d(noise_dir)),
                            C.c_double(strength), C.c_double(frequency))
    return cams, pts


def total_reprojection_error(cams, pts, offsets, point_idx, uv, norm):
    cams, pts, uv = _d(cams).reshape(-1), _d(pts).reshape(-1), _d(uv).reshape(-1)
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    idx = np.ascontiguousarray(point_idx, dtype=np.uint64)
    return float(lib().orc_total_reprojection_error(
        _p(cams), _u64(cams.size // CAM), _p(pts), _p(off, C.c_uint64), _p(idx, C.c_uint64),
        _p(uv), C.c_double(norm)))
