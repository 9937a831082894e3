"""Host mirror of city2ba::baproblem (reference: src/baproblem.rs).

SnavelyCamera math goes through the C ABI's host helpers (same arithmetic order as the device
code); BAProblem keeps cameras as a (C,15) record array, points as (P,3) and the visibility graph
as CSR.  Graph post-processing (`cull`) and BAL I/O are host code, as in the reference.
"""
from __future__ import annotations

import ctypes as C
import math
import struct

import numpy as np

from ._lib import CAM_STRIDE, check, context, lib
from .generate import VisGraph

_pd = C.POINTER(C.c_double)


def _p(a):
    return a.ctypes.data_as(_pd)


class Error(Exception):
    """city2ba::Error (src/baproblem.rs:32-62)."""


class ParseError(Error):
    pass


class EmptyProblem(Error):
    pass


class IOError_(Error):
    pass


# ---- rotations in cgmath's conventions (column-major 3x3 flattened to 9) ----------------------
def from_angle_y(rad):
    s, c = math.sin(rad), math.cos(rad)
    return np.array([c, 0, -s, 0, 1, 0, s, 0, c], dtype=np.float64)


def from_angle_x(rad):
    s, c = math.sin(rad), math.cos(rad)
    return np.array([1, 0, 0, 0, c, s, 0, -s, c], dtype=np.float64)


def from_axis_angle(axis, rad):
    s, c = math.sin(rad), math.cos(rad)
    k = 1.0 - c
    x, y, z = (float(v) for v in axis)
    return np.array([k * x * x + c, k * x * y + s * z, k * x * z - s * y,
                     k * x * y - s * z, k * y * y + c, k * y * z + s * x,
                     k * x * z + s * y, k * y * z - s * x, k * z * z + c], dtype=np.float64)


def _quat_from_mat(m):
    M = lambda c, r: m[c * 3 + r]  # noqa: E731
    trace = (M(0, 0) + M(1, 1)) + M(2, 2)
    if trace >= 0.0:
        s = math.sqrt(1.0 + trace)
        w = 0.5 * s
        s = 0.5 / s
        return w, (M(1, 2) - M(2, 1)) * s, (M(2, 0) - M(0, 2)) * s, (M(0, 1) - M(1, 0)) * s
    if M(0, 0) > M(1, 1) and M(0, 0) > M(2, 2):
        s = math.sqrt(((M(0, 0) - M(1, 1)) - M(2, 2)) + 1.0)
        x = 0.5 * s
        s = 0.5 / s
        return (M(1, 2) - M(2, 1)) * s, x, (M(1, 0) + M(0, 1)) * s, (M(0, 2) + M(2, 0)) * s
    if M(1, 1) > M(2, 2):
        s = math.sqrt(((M(1, 1) - M(0, 0)) - M(2, 2)) + 1.0)
        y = 0.5 * s
        s = 0.5 / s
        return (M(2, 0) - M(0, 2)) * s, (M(1, 0) + M(0, 1)) * s, y, (M(2, 1) + M(1, 2)) * s
    s = math.sqrt(((M(2, 2) - M(0, 0)) - M(1, 1)) + 1.0)
    z = 0.5 * s
    s = 0.5 / s
    return (M(0, 1) - M(1, 0)) * s, (M(0, 2) + M(2, 0)) * s, (M(2, 1) + M(1, 2)) * s, z


def _mat_from_quat(q):
    s, x, y, z = q
    x2, y2, z2 = x + x, y + y, z + z
    xx2, xy2, xz2 = x2 * x, x2 * y, x2 * z
    yy2, yz2, zz2 = y2 * y, y2 * z, z2 * z
    sy2, sz2, sx2 = y2 * s, z2 * s, x2 * s
    return np.array([1.0 - yy2 - zz2, xy2 + sz2, xz2 - sy2, xy2 - sz2, 1.0 - xx2 - zz2, yz2 + sx2,
                     xz2 + sy2, yz2 - sx2, 1.0 - xx2 - yy2], dtype=np.float64)


def _ulps_eq(a, b):
    """approx::ulps_eq! with its defaults (epsilon = f64::EPSILON, max_ulps = 4), as cgmath 0.17 uses it"""
    if abs(a - b) <= 2.220446049250313e-16:
        return True
    if math.copysign(1.0, a) != math.copysign(1.0, b):
        return False
    ia, ib = (int(np.float64(x).view(np.int64)) for x in (a, b))
    return abs(ia - ib) <= 4


def between_vectors(a, b):
    """cgmath 0.17 Basis3::between_vectors (through Quaternion::between_vectors), used by the path cameras
    (src/generate.rs:144,200): column-major 3x3 as 9 doubles"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    k_cos_theta = float(a @ b)
    if _ulps_eq(k_cos_theta, 1.0):
        return np.array([1, 0, 0, 0, 1, 0, 0, 0, 1], np.float64)
    k = math.sqrt(float(a @ a) * float(b @ b))
    if _ulps_eq(k_cos_theta / k, -1.0):
        o = np.cross([1.0, 0.0, 0.0], a)
        if _ulps_eq(float(o @ o), 0.0):
            o = np.cross([0.0, 1.0, 0.0], a)
        o = o / np.linalg.norm(o)
        return _mat_from_quat(np.array([0.0, o[0], o[1], o[2]]))
    q = np.concatenate([[k + k_cos_theta], np.cross(a, b)])
    return _mat_from_quat(q / np.linalg.norm(q))


def from_rodrigues(v):
    """src/baproblem.rs:78-90"""
    x = [float(t) for t in v]
    theta2 = (x[0] * x[0] + x[1] * x[1]) + x[2] * x[2]
    if theta2 > 2.220446049250313e-16:
        angle = math.sqrt(theta2)
        inv = 1.0 / angle
        return from_axis_angle([x[0] * inv, x[1] * inv, x[2] * inv], angle)
    m = [1.0, x[2], -x[1], -x[2], 1.0, x[0], x[1], -x[0], 1.0]
    return _mat_from_quat(_quat_from_mat(m))


def to_rodrigues(R):
    """src/baproblem.rs:93-102"""
    q = _quat_from_mat([float(t) for t in R])
    angle = 2.0 * math.acos(max(-1.0, min(1.0, q[0])))
    d = 1.0 - q[0] * q[0]
    if d < 2.220446049250313e-16:
        return np.zeros(3)
    sd = math.sqrt(d)
    a = np.array([q[1] / sd, q[2] / sd, q[3] / sd])
    n = a * (1.0 / math.sqrt((a[0] * a[0] + a[1] * a[1]) + a[2] * a[2]))
    return n * angle


class SnavelyCamera:
    """Camera expressed as Rx+t with intrinsics; looks down -z, +y up (src/baproblem.rs:127-176)."""

    __slots__ = ("rec",)

    def __init__(self, loc=None, dir=None, intrin=None, record=None):
        if record is not None:
            self.rec = np.array(record, dtype=np.float64).reshape(CAM_STRIDE)
        else:
            self.rec = np.empty(CAM_STRIDE)
            self.rec[0:9] = np.asarray(dir, dtype=np.float64).reshape(9)
            self.rec[9:12] = loc
            self.rec[12:15] = intrin if intrin is not None else (1.0, 0.0, 0.0)

    # field views
    @property
    def dir(self):
        return self.rec[0:9]

    @property
    def loc(self):
        return self.rec[9:12]

    @property
    def intrin(self):
        return self.rec[12:15]

    def to_record(self):
        return self.rec

    def project_world(self, p):
        p = np.ascontiguousarray(p, np.float64)
        out = np.empty(3)
        lib().c2b_camera_project_world(_p(self.rec), _p(p), _p(out))
        return out

    def project(self, pc):
        pc = np.ascontiguousarray(pc, np.float64)
        out = np.empty(2)
        lib().c2b_camera_project(_p(self.rec), _p(pc), _p(out))
        return out

    @classmethod
    def from_position_direction(cls, position, dir):
        pos = np.ascontiguousarray(position, np.float64)
        R = np.ascontiguousarray(dir, np.float64).reshape(9)
        out = np.empty(CAM_STRIDE)
        lib().c2b_camera_from_position_direction(_p(pos), _p(R), _p(out))
        return cls(record=out)

    def center(self):
        out = np.empty(3)
        lib().c2b_camera_center(_p(self.rec), _p(out))
        return out

    def transform(self, delta_dir, delta_loc):
        dR = np.ascontiguousarray(delta_dir, np.float64).reshape(9)
        dl = np.ascontiguousarray(delta_loc, np.float64)
        out = np.empty(CAM_STRIDE)
        lib().c2b_camera_transform(_p(self.rec), _p(dR), _p(dl), _p(out))
        return SnavelyCamera(record=out)

    def to_world(self, p):
        """dir.invert().rotate_point(p - loc), src/baproblem.rs:173-175"""
        R = self.rec[0:9].reshape(3, 3).T  # row-major view of the column-major matrix
        return np.linalg.inv(R) @ (np.asarray(p, np.float64) - self.loc)

    @classmethod
    def from_vec(cls, x):
        x = [float(t) for t in x]
        return cls(loc=x[3:6], dir=from_rodrigues(x[0:3]), intrin=x[6:9])

    def to_vec(self):
        return np.concatenate([to_rodrigues(self.dir), self.loc, self.intrin])

    def rotation(self):
        return self.dir

    def focal_length(self):
        return float(self.rec[12])

    def distortion(self):
        return float(self.rec[13]), float(self.rec[14])

    def modify_intrin(self, delta):
        r = self.rec.copy()
        r[12:15] += np.asarray(delta, np.float64)
        return SnavelyCamera(record=r)


def _project_all(cams, pts, offsets, point_idx):
    """vectorised SnavelyCamera::project(project_world(p)) for every observation (numpy f64)."""
    counts = np.diff(offsets.astype(np.int64))
    cam_of = np.repeat(np.arange(len(counts)), counts)
    c = cams[cam_of]
    p = pts[point_idx.astype(np.int64)]
    pc = np.empty_like(p)
    for r in range(3):
        pc[:, r] = ((c[:, 0 + r] * p[:, 0] + c[:, 3 + r] * p[:, 1]) + c[:, 6 + r] * p[:, 2]) + c[:, 9 + r]
    with np.errstate(divide="ignore", invalid="ignore"):
        px, py = -pc[:, 0] / pc[:, 2], -pc[:, 1] / pc[:, 2]
    m2 = px * px + py * py
    r = (1.0 + c[:, 13] * m2) + c[:, 14] * (m2 * m2)
    fr = c[:, 12] * r
    return np.stack([fr * px, fr * py], axis=1)


class BAProblem:
    """Bundle adjustment problem (src/baproblem.rs:251-260): cameras, points, visibility graph."""

    def __init__(self, cameras, points, vis_graph: VisGraph):
        self.cameras = np.ascontiguousarray(cameras, np.float64).reshape(-1, CAM_STRIDE)
        self.points = np.ascontiguousarray(points, np.float64).reshape(-1, 3)
        self.vis_graph = vis_graph

    # ---- constructors --------------------------------------------------------------------------
    @classmethod
    def from_visibility(cls, cams, points, obs):
        """src/baproblem.rs:360-376: asserts len(obs) == cameras and indices in range."""
        from .generate import _cam_array
        cams = _cam_array(cams)
        points = np.ascontiguousarray(points, np.float64).reshape(-1, 3)
        if not isinstance(obs, VisGraph):
            offsets = np.zeros(len(obs) + 1, np.uint64)
            idx, uv = [], []
            for i, o in enumerate(obs):
                offsets[i + 1] = offsets[i] + len(o)
                for p, (u, v) in o:
                    idx.append(p)
                    uv.append((u, v))
            obs = VisGraph(offsets, np.array(idx, np.uint64), np.array(uv, np.float64).reshape(-1, 2))
        assert len(cams) == len(obs), "cams.len() == obs.len()"
        if obs.num_observations:
            assert int(obs.point_idx.max()) < len(points), "observation references a missing point"
        return cls(cams, points, obs)

    @classmethod
    def new(cls, cams, points, obs):
        """src/baproblem.rs:342-355: obs = iterable of (camera, point, u, v)."""
        from .generate import _cam_array
        cams = _cam_array(cams)
        per = [[] for _ in range(len(cams))]
        for ci, pi, u, v in obs:
            assert ci < len(cams) and pi < len(points)
            per[ci].append((pi, (u, v)))
        return cls.from_visibility(cams, points, per)

    # ---- sizes ---------------------------------------------------------------------------------
    def num_points(self):
        return len(self.points)

    def num_cameras(self):
        return len(self.cameras)

    def num_observations(self):
        return self.vis_graph.num_observations

    def __str__(self):
        return ("Bundle Adjustment Problem with {} cameras, {} points, and {} observations".format(
            self.num_cameras(), self.num_points(), self.num_observations()))

    # ---- statistics ----------------------------------------------------------------------------
    def total_reprojection_error(self, norm: float) -> float:
        """src/baproblem.rs:265-279"""
        g = self.vis_graph
        if g.num_observations == 0:
            return 0.0
        q = _project_all(self.cameras, self.points, g.offsets, g.point_idx)
        d = np.abs(q - g.uv)
        return float(np.sum(d ** norm) ** (1.0 / norm))

    def mean_std(self, ctx=None):
        """BAProblem::mean / std (src/baproblem.rs:282-304) as GPU tree reductions."""
        ctx = ctx or context()
        m, s = np.empty(3), np.empty(3)
        check(lib().c2b_mean_std(ctx.handle, _p(self.cameras), len(self.cameras), _p(self.points),
                                 len(self.points), _p(m), _p(s)))
        return m, s

    def mean(self):
        return self.mean_std()[0]

    def std(self):
        return self.mean_std()[1]

    def centers(self):
        out = np.empty((len(self.cameras), 3))
        for i, c in enumerate(self.cameras):
            lib().c2b_camera_center(_p(np.ascontiguousarray(c)), _p(out[i]))
        return out

    def extent(self):
        """src/baproblem.rs:307-331"""
        allp = np.concatenate([self.centers(), self.points])
        return allp.min(axis=0), allp.max(axis=0)

    def dimensions(self):
        lo, hi = self.extent()
        return hi - lo

    # ---- graph post-processing (host, as in the reference) ----------------------------------------
    def subset(self, ci, pi):
        """src/baproblem.rs:394-423"""
        ci = np.asarray(ci, np.int64)
        pi = np.asarray(pi, np.int64)
        g = self.vis_graph
        remap = np.full(len(self.points), -1, np.int64)
        remap[pi] = np.arange(len(pi))
        counts = g.counts()
        cam_of = np.repeat(np.arange(len(counts)), counts)
        cam_keep = np.zeros(len(self.cameras), bool)
        cam_keep[ci] = True
        new_pt = remap[g.point_idx.astype(np.int64)]
        keep = cam_keep[cam_of] & (new_pt >= 0)
        cam_new = np.full(len(self.cameras), -1, np.int64)
        cam_new[ci] = np.arange(len(ci))
        kc = cam_new[cam_of[keep]]
        order = np.argsort(kc, kind="stable")
        new_counts = np.bincount(kc, minlength=len(ci))
        offsets = np.zeros(len(ci) + 1, np.uint64)
        offsets[1:] = np.cumsum(new_counts)
        return BAProblem(self.cameras[ci], self.points[pi],
                         VisGraph(offsets, new_pt[keep][order].astype(np.uint64), g.uv[keep][order]))

    def remove_singletons(self):
        """src/baproblem.rs:426-453: cameras need > 3 observations, points > 1."""
        g = self.vis_graph
        ci = np.nonzero(g.counts() > 3)[0]
        pc = np.bincount(g.point_idx.astype(np.int64), minlength=len(self.points))
        pi = np.nonzero(pc > 1)[0]
        return self.subset(ci, pi)

    def largest_connected_component(self):
        """src/baproblem.rs:456-534 (union-find over cameras + points; largest set wins; ties are
        hash-map order in the reference, lowest label here).  Kept as written there, including the
        observation filter at :523 that looks up sets[point index] WITHOUT the camera offset: an
        observation of point i by a camera of the component is dropped when entity i of the combined
        (cameras, then points) numbering lies outside the component."""
        if self.num_cameras() == 0:
            return self
        from scipy.sparse import coo_matrix
        from scipy.sparse.csgraph import connected_components
        g = self.vis_graph
        nc, npt = self.num_cameras(), self.num_points()
        counts = g.counts()
        cam_of = np.repeat(np.arange(nc), counts)
        n = nc + npt
        idx = g.point_idx.astype(np.int64)
        A = coo_matrix((np.ones(len(cam_of), np.int8), (cam_of, idx + nc)), shape=(n, n))
        _, labels = connected_components(A, directed=False)
        sizes = np.bincount(labels)
        lcc = int(np.argmax(sizes))
        ci = np.nonzero(labels[:nc] == lcc)[0]
        pi = np.nonzero(labels[nc:] == lcc)[0]
        keep = labels[idx] == lcc                          # the reference's sets[x.0] (no + num_cameras)
        if not np.all(keep):
            new_counts = np.bincount(cam_of[keep], minlength=nc)
            offsets = np.zeros(nc + 1, np.uint64)
            offsets[1:] = np.cumsum(new_counts)
            filtered = BAProblem(self.cameras, self.points, VisGraph(offsets, g.point_idx[keep], g.uv[keep]))
            return filtered.subset(ci, pi)
        return self.subset(ci, pi)

    def cull_gpu(self, ctx=None, stats=None):
        """cull() on the GPU (c2b_cull_problem): the same problem, bit for bit.  Works on copies; `stats`, a dict
        if given, receives the call's c2b_cull_stats (iterations, device times)."""
        from ._lib import CullStats
        ctx = ctx or context()
        g = self.vis_graph
        cams = np.array(self.cameras, np.float64, order="C").reshape(-1, CAM_STRIDE)
        pts = np.array(self.points, np.float64, order="C").reshape(-1, 3)
        off = np.array(g.offsets, np.uint64, order="C")
        if len(off) != len(cams) + 1:
            raise ValueError("cameras and CSR offsets disagree")
        idx = g.point_idx
        if len(idx) and int(idx.max()) > 0xffffffff:
            raise ValueError("point index does not fit 32 bits")
        idx = np.array(idx, np.uint32, order="C")
        uv = np.array(g.uv, np.float64, order="C").reshape(-1, 2)
        st = CullStats()
        check(lib().c2b_cull_problem(ctx.handle, _p(cams), len(cams), _p(pts), len(pts),
                                     off.ctypes.data_as(C.POINTER(C.c_uint64)),
                                     idx.ctypes.data_as(C.POINTER(C.c_uint32)), _p(uv), C.byref(st)))
        if stats is not None:
            stats.update(st.to_dict())
        nc, npt, no = int(st.n_cameras), int(st.n_points), int(st.n_obs)
        return BAProblem(cams[:nc].copy(), pts[:npt].copy(),
                         VisGraph(off[:nc + 1].copy(), idx[:no].astype(np.uint64), uv[:no].copy()))

    def cull(self):
        """src/baproblem.rs:538-549: iterate LCC then remove_singletons to a fixed point."""
        nc, npt = self.num_cameras(), self.num_points()
        culled = self.largest_connected_component().remove_singletons()
        while culled.num_cameras() != nc or culled.num_points() != npt:
            nc, npt = culled.num_cameras(), culled.num_points()
            culled = culled.largest_connected_component().remove_singletons()
        return culled

    # ---- BAL I/O (src/baproblem.rs:580-785) --------------------------------------------------------
    def _camera_vecs(self):
        return np.stack([SnavelyCamera(record=c).to_vec() for c in self.cameras]) \
            if len(self.cameras) else np.zeros((0, 9))

    def write_binary(self, path):
        """src/baproblem.rs:736-764: big-endian u64/f64, per-camera count-prefixed lists."""
        g = self.vis_graph
        with open(path, "wb") as f:
            f.write(struct.pack(">QQQ", self.num_cameras(), self.num_points(), g.num_observations))
            rec = np.empty(g.num_observations, dtype=[("p", ">u8"), ("u", ">f8"), ("v", ">f8")])
            rec["p"], rec["u"], rec["v"] = g.point_idx, g.uv[:, 0], g.uv[:, 1]
            for c in range(self.num_cameras()):
                a, b = int(g.offsets[c]), int(g.offsets[c + 1])
                f.write(struct.pack(">Q", b - a))
                f.write(rec[a:b].tobytes())
            f.write(self._camera_vecs().astype(">f8").tobytes())
            f.write(self.points.astype(">f8").tobytes())

    def write_text(self, path):
        """src/baproblem.rs:709-733 (Rust `{}` prints the shortest round-trip decimal, never an
        exponent; Python's repr is the same shortest digits, expanded to positional form)."""
        g = self.vis_graph
        fmt = lambda x: np.format_float_positional(x, trim="-", unique=True)  # noqa: E731
        counts = g.counts()
        cam_of = np.repeat(np.arange(len(counts)), counts)
        with open(path, "w") as f:
            f.write(f"{self.num_cameras()} {self.num_points()} {g.num_observations}\n")
            for c, p, (u, v) in zip(cam_of, g.point_idx, g.uv):
                f.write(f"{c} {int(p)} {fmt(u)} {fmt(v)}\n")
            for v in self._camera_vecs():
                f.write(" ".join(fmt(x) for x in v) + "\n")
            for p in self.points:
                f.write(f"{fmt(p[0])} {fmt(p[1])} {fmt(p[2])}\n")

    @staticmethod
    def _bal_binary(path):
        """src/baproblem.rs:768-785: the extension picks the format (True: .bbal, False: .bal)"""
        path = str(path)
        if "." not in path.rsplit("/", 1)[-1]:
            raise IOError_("file does not have an extension")
        ext = path.rsplit(".", 1)[-1]
        if ext not in ("bal", "bbal"):
            raise IOError_(f"unknown file extension {ext}")
        return ext == "bbal"

    def write(self, path):
        """src/baproblem.rs:768-785"""
        return self.write_binary(path) if self._bal_binary(path) else self.write_text(path)

    def write_gpu(self, path, ctx=None, stats=None):
        """write() with the file encoded on the GPU (c2b_write_bal) and streamed to disk in chunks.  The bytes are
        the reference's: the shortest round-trip digits of every value, positional, camera vectors from the host's
        to_vec (c2b_camera_to_vec).  `stats`, a dict if given, receives bytes, chunks and the encode / D2H / write
        times."""
        from ._lib import C2BError, BalStats, BAL_BINARY, BAL_TEXT, ERR_IO
        fmt = BAL_BINARY if self._bal_binary(path) else BAL_TEXT
        ctx = ctx or context()
        g = self.vis_graph
        cams = np.ascontiguousarray(self.cameras, np.float64).reshape(-1, CAM_STRIDE)
        pts = np.ascontiguousarray(self.points, np.float64).reshape(-1, 3)
        off = np.ascontiguousarray(g.offsets, np.uint64)
        if len(off) != len(cams) + 1:
            raise ValueError("cameras and CSR offsets disagree")
        idx = g.point_idx
        if len(idx) and int(idx.max()) > 0xffffffff:
            raise ValueError("point index does not fit 32 bits")
        idx = np.ascontiguousarray(idx, np.uint32)
        uv = np.ascontiguousarray(g.uv, np.float64).reshape(-1, 2)
        st = BalStats()
        try:
            check(lib().c2b_write_bal(ctx.handle, str(path).encode(), fmt, _p(cams), len(cams), _p(pts), len(pts),
                                      off.ctypes.data_as(C.POINTER(C.c_uint64)),
                                      idx.ctypes.data_as(C.POINTER(C.c_uint32)), _p(uv), C.byref(st)))
        except C2BError as e:
            if e.code == ERR_IO:
                raise IOError_(str(e)) from e
            raise
        if stats is not None:
            stats.update(st.to_dict())

    @classmethod
    def from_file_binary(cls, path):
        """src/baproblem.rs:632-693"""
        data = open(path, "rb").read()
        try:
            nc, npt, _ = struct.unpack_from(">QQQ", data, 0)
            off = 24
            offsets = np.zeros(nc + 1, np.uint64)
            chunks = []
            for c in range(nc):
                (n,) = struct.unpack_from(">Q", data, off)
                off += 8
                chunks.append(np.frombuffer(data, dtype=[("p", ">u8"), ("u", ">f8"), ("v", ">f8")],
                                            count=n, offset=off))
                off += 24 * n
                offsets[c + 1] = offsets[c] + n
            rec = np.concatenate(chunks) if chunks else np.zeros(0, dtype=[("p", ">u8"), ("u", ">f8"), ("v", ">f8")])
            cams9 = np.frombuffer(data, dtype=">f8", count=9 * nc, offset=off).reshape(nc, 9)
            off += 72 * nc
            pts = np.frombuffer(data, dtype=">f8", count=3 * npt, offset=off).reshape(npt, 3)
        except (struct.error, ValueError) as e:
            raise ParseError("Binary parse error") from e
        cams = np.stack([SnavelyCamera.from_vec(v).rec for v in cams9]) if nc else np.zeros((0, CAM_STRIDE))
        uv = np.stack([rec["u"], rec["v"]], axis=1).astype(np.float64)
        return cls(cams, pts.astype(np.float64), VisGraph(offsets, rec["p"].astype(np.uint64), uv))

    @classmethod
    def from_file_text(cls, path):
        """src/baproblem.rs:580-628 (any whitespace separates tokens)."""
        tok = open(path).read().split()
        try:
            def digits(t):  # nom's digit1: an index is digits only ("-1", "1.5", "1e3" are parse errors)
                if not t.isdigit():
                    raise ValueError(f"not an unsigned integer: {t!r}")
                return int(t)
            nc, npt, no = digits(tok[0]), digits(tok[1]), digits(tok[2])
            if 4 * no + 9 * nc + 3 * npt > len(tok) - 3:
                raise ValueError("header counts exceed the file")
            ci = [digits(t) for t in tok[3:3 + 4 * no:4]]
            pi = [digits(t) for t in tok[4:3 + 4 * no:4]]
            ou = np.array(tok[5:3 + 4 * no:4], dtype=np.float64)
            ov = np.array(tok[6:3 + 4 * no:4], dtype=np.float64)
            base = 3 + 4 * no
            cams9 = np.array(tok[base:base + 9 * nc], dtype=np.float64).reshape(nc, 9)
            base += 9 * nc
            pts = np.array(tok[base:base + 3 * npt], dtype=np.float64).reshape(npt, 3)
        except (ValueError, IndexError) as e:
            raise ParseError(str(e)) from e
        cams = np.stack([SnavelyCamera.from_vec(v).rec for v in cams9]) if nc else np.zeros((0, CAM_STRIDE))
        return cls.new(cams, pts, list(zip(ci, pi, ou.tolist(), ov.tolist())))

    @classmethod
    def from_file_gpu(cls, path, ctx=None, stats=None):
        """from_file() with the file parsed on the GPU (c2b_read_bal_resident), then the problem and its CSR
        downloaded.  The file's problem REPLACES the ctx's resident problem.  Raises what from_file raises: ParseError,
        IOError_, AssertionError for an observation index out of range.  `stats`, a dict if given, receives the read's
        stats (bytes, chunks, slow_tokens, regrouped, ms_read, ms_h2d, ms_parse)."""
        from .generate import ResidentProblem
        rp = ResidentProblem(ctx or context())
        st = rp.read(path)
        if stats is not None:
            stats.update(st)
        cams, pts = rp.download_problem(st["n_cameras"], st["n_points"])
        g = rp.download()
        return cls(cams, pts, VisGraph(g.offsets, g.point_idx.astype(np.uint64), g.uv.reshape(-1, 2)))

    @classmethod
    def from_file(cls, path):
        """src/baproblem.rs:697-706"""
        ext = str(path).rsplit(".", 1)[-1]
        if ext == "bal":
            return cls.from_file_text(path)
        if ext == "bbal":
            return cls.from_file_binary(path)
        raise IOError_(f"unknown file extension {ext}")
