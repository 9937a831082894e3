"""ctypes binding of libcity2ba_cuda.so (the C ABI in include/city2ba_cuda.h).

The library is the product: there is no CPU fallback.  Importing this module fails loudly when
the shared object is missing (run `python -c "import __graft_entry__ as g; g.build()"`), and
`context()` fails loudly when no sm_100 GPU is visible.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libcity2ba_cuda.so")

CAM_STRIDE = 15


class C2BError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"city2ba_cuda error {code}: {msg}")
        self.code = code


class VisOptions(C.Structure):
    _fields_ = [
        ("cull_mode", C.c_int),
        ("occlusion", C.c_int),
        ("endpoint_guard_rel", C.c_int),
        ("count_traversal", C.c_int),
        ("block_length", C.c_double),
        ("block_inset", C.c_double),
        ("predicate", C.c_int),
        ("reserved", C.c_int),
    ]


class Obs(C.Structure):
    _fields_ = [
        ("n_cameras", C.c_uint64),
        ("n_obs", C.c_uint64),
        ("offsets", C.POINTER(C.c_uint64)),
        ("point_idx", C.POINTER(C.c_uint32)),
        ("uv", C.POINTER(C.c_double)),
        ("n_candidates", C.c_uint64),
        ("pairs_evaluated", C.c_uint64),
        ("nodes_visited", C.c_uint64),
        ("tris_tested", C.c_uint64),
        ("h2d_bytes", C.c_uint64),
        ("d2h_bytes", C.c_uint64),
        ("ms_h2d", C.c_float),
        ("ms_prep", C.c_float),
        ("ms_cull", C.c_float),
        ("ms_sort", C.c_float),
        ("ms_traverse", C.c_float),
        ("ms_compact", C.c_float),
        ("ms_d2h", C.c_float),
        ("ms_total", C.c_float),
    ]


class Ray48(C.Structure):
    _fields_ = [
        ("org_x", C.c_float), ("org_y", C.c_float), ("org_z", C.c_float), ("tnear", C.c_float),
        ("dir_x", C.c_float), ("dir_y", C.c_float), ("dir_z", C.c_float), ("time", C.c_float),
        ("tfar", C.c_float), ("mask", C.c_uint32), ("id", C.c_uint32), ("flags", C.c_uint32),
    ]


MAX_GPUS = 16


class MultiStats(C.Structure):
    _fields_ = [
        ("n_gpus", C.c_int),
        ("cam_begin", C.c_uint64 * MAX_GPUS), ("cam_end", C.c_uint64 * MAX_GPUS),
        ("n_obs", C.c_uint64 * MAX_GPUS), ("obs_base", C.c_uint64 * MAX_GPUS),
        ("ms_points", C.c_float * MAX_GPUS), ("ms_compute", C.c_float * MAX_GPUS),
        ("ms_exchange", C.c_float * MAX_GPUS), ("ms_d2h", C.c_float * MAX_GPUS),
        ("ms_wall", C.c_float),
    ]


class CullStats(C.Structure):
    """c2b_cull_stats: sizes after LCC + remove_singletons to a fixed point, and device times"""
    _fields_ = [
        ("n_cameras", C.c_uint64), ("n_points", C.c_uint64), ("n_obs", C.c_uint64),
        ("iterations", C.c_uint32), ("reserved", C.c_uint32),
        ("ms_h2d", C.c_float), ("ms_compute", C.c_float), ("ms_d2h", C.c_float),
    ]

    def to_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class MismatchStats(C.Structure):
    """c2b_mismatch_stats: selected observations, those whose partner is another observation, and device times"""
    _fields_ = [
        ("n_selected", C.c_uint64), ("n_swapped", C.c_uint64),
        ("ms_h2d", C.c_float), ("ms_compute", C.c_float), ("ms_d2h", C.c_float),
    ]

    def to_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class BalStats(C.Structure):
    """c2b_bal_stats: bytes and chunks of one BAL file, device ms of encode / D2H, host ms of write(2)"""
    _fields_ = [
        ("bytes", C.c_uint64), ("chunks", C.c_uint64),
        ("ms_encode", C.c_float), ("ms_d2h", C.c_float), ("ms_write", C.c_float),
    ]

    def to_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class BalReadStats(C.Structure):
    """c2b_bal_read_stats: sizes, bytes and chunks read, tokens converted on the host, whether the observations were
    regrouped by camera, host ms in pread(2), device ms of the chunk copies and of the parse kernels"""
    _fields_ = [
        ("n_cameras", C.c_uint64), ("n_points", C.c_uint64), ("n_obs", C.c_uint64),
        ("bytes", C.c_uint64), ("chunks", C.c_uint64), ("slow_tokens", C.c_uint64),
        ("regrouped", C.c_uint32), ("reserved", C.c_uint32),
        ("ms_read", C.c_float), ("ms_h2d", C.c_float), ("ms_parse", C.c_float),
    ]

    def to_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


CULL_GRID, CULL_EXHAUSTIVE = 0, 1
BAL_TEXT, BAL_BINARY = 0, 1
ERR_INVALID, ERR_IO, ERR_PARSE = -1, -7, -8
OCC_MESH, OCC_NONE, OCC_ANALYTIC = 0, 1, 2
PRED_WATERTIGHT, PRED_MT = 0, 1

# every symbol include/city2ba_cuda.h declares
EXPORTS = [
    "c2b_init", "c2b_shutdown", "c2b_last_error", "c2b_abi_version", "c2b_kernel_launches", "c2b_probe_fp64",
    "c2b_scene_create", "c2b_scene_bounds", "c2b_scene_num_triangles", "c2b_scene_num_nodes",
    "c2b_scene_destroy", "c2b_occluded", "c2b_intersect", "c2b_intersect1", "c2b_vis_options_default",
    "c2b_visibility_graph", "c2b_obs_free", "c2b_upload_points", "c2b_upload_points_device", "c2b_upload_cameras", "c2b_drop_point_grid",
    "c2b_tune", "c2b_points_device_buffer", "c2b_points_commit", "c2b_download_obs_into",
    "c2b_init_multi", "c2b_shutdown_multi", "c2b_multi_num_gpus", "c2b_multi_ctx", "c2b_scene_create_multi",
    "c2b_scene_destroy_multi", "c2b_multi_scene_get", "c2b_visibility_graph_multi",
    "c2b_visibility_graph_resident", "c2b_download_obs", "c2b_reprojection_error_resident",
    "c2b_add_drift", "c2b_add_drift_normalized", "c2b_add_noise", "c2b_add_sin_noise", "c2b_noise_timing",
    "c2b_add_drift_resident", "c2b_add_noise_resident", "c2b_add_sin_noise_resident", "c2b_download_problem",
    "c2b_mean_std", "c2b_cull_problem", "c2b_cull_problem_resident",
    "c2b_add_incorrect_correspondences", "c2b_add_incorrect_correspondences_resident", "c2b_write_bal", "c2b_write_bal_resident",
    "c2b_read_bal_resident", "c2b_generate_world_points_uniform",
    "c2b_grid_num_cameras", "c2b_grid_num_points", "c2b_grid_cameras", "c2b_grid_points",
    "c2b_line_cameras", "c2b_line_points", "c2b_city_mesh", "c2b_camera_center",
    "c2b_camera_project_world", "c2b_camera_project", "c2b_camera_from_position_direction",
    "c2b_camera_transform", "c2b_camera_to_vec", "c2b_camera_from_vec",
]

_lib = None


def lib():
    """Load the shared library (no GPU needed for loading or for the host-only entry points)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(
            f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a).  city2ba_b200 has no CPU fallback.")
    L = C.CDLL(SO_PATH)
    vp, u64, dbl, i32 = C.c_void_p, C.c_uint64, C.c_double, C.c_int
    pd, pf, pu32 = C.POINTER(C.c_double), C.POINTER(C.c_float), C.POINTER(C.c_uint32)
    L.c2b_last_error.restype = C.c_char_p
    L.c2b_kernel_launches.restype = u64
    L.c2b_init.argtypes = [i32, C.POINTER(vp)]
    L.c2b_shutdown.argtypes = [vp]
    L.c2b_shutdown.restype = None
    L.c2b_scene_create.argtypes = [vp, pf, u64, pu32, u64, C.POINTER(vp)]
    L.c2b_scene_bounds.argtypes = [vp, pf, pf]
    L.c2b_scene_num_triangles.argtypes = [vp]
    L.c2b_scene_num_triangles.restype = u64
    L.c2b_scene_num_nodes.argtypes = [vp]
    L.c2b_scene_num_nodes.restype = u64
    L.c2b_scene_destroy.argtypes = [vp]
    L.c2b_scene_destroy.restype = None
    L.c2b_occluded.argtypes = [vp, vp, C.POINTER(Ray48), u64]
    L.c2b_intersect.argtypes = [vp, vp, C.POINTER(Ray48), u64]
    L.c2b_intersect1.argtypes = [vp, vp, pf, pf, C.POINTER(i32), pf]
    L.c2b_vis_options_default.argtypes = [C.POINTER(VisOptions)]
    L.c2b_vis_options_default.restype = None
    L.c2b_visibility_graph.argtypes = [vp, vp, vp, u64, vp, u64, dbl, C.POINTER(VisOptions),
                                       C.POINTER(Obs)]
    L.c2b_obs_free.argtypes = [vp, C.POINTER(Obs)]
    L.c2b_obs_free.restype = None
    L.c2b_upload_points.argtypes = [vp, vp, u64]
    L.c2b_upload_points_device.argtypes = [vp, vp, u64]
    L.c2b_upload_cameras.argtypes = [vp, vp, u64]
    L.c2b_drop_point_grid.argtypes = [vp]
    L.c2b_tune.argtypes = [vp, C.c_char_p, dbl]
    L.c2b_points_device_buffer.argtypes = [vp, u64, C.POINTER(vp)]
    L.c2b_points_commit.argtypes = [vp, u64]
    L.c2b_download_obs_into.argtypes = [vp, u64, vp, vp, vp, i32, pf]
    L.c2b_init_multi.argtypes = [i32, C.POINTER(i32), C.POINTER(vp)]
    L.c2b_shutdown_multi.argtypes = [vp]
    L.c2b_shutdown_multi.restype = None
    L.c2b_multi_num_gpus.argtypes = [vp]
    L.c2b_multi_ctx.argtypes = [vp, i32]
    L.c2b_multi_ctx.restype = vp
    L.c2b_scene_create_multi.argtypes = [vp, pf, u64, pu32, u64, C.POINTER(vp)]
    L.c2b_scene_destroy_multi.argtypes = [vp]
    L.c2b_multi_scene_get.argtypes = [vp, i32]
    L.c2b_multi_scene_get.restype = vp
    L.c2b_scene_destroy_multi.restype = None
    L.c2b_visibility_graph_multi.argtypes = [vp, vp, vp, u64, vp, u64, dbl, C.POINTER(VisOptions), C.POINTER(Obs),
                                             C.POINTER(MultiStats)]
    L.c2b_visibility_graph_resident.argtypes = [vp, vp, dbl, C.POINTER(VisOptions), C.POINTER(Obs)]
    L.c2b_download_obs.argtypes = [vp, C.POINTER(Obs)]
    L.c2b_reprojection_error_resident.argtypes = [vp, dbl, pd]
    L.c2b_add_drift.argtypes = [vp, pd, u64, pd, u64, dbl, dbl, dbl, pd, u64]
    L.c2b_add_drift_normalized.argtypes = [vp, pd, u64, pd, u64, dbl, dbl, dbl, u64]
    L.c2b_add_noise.argtypes = [vp, pd, u64, pd, u64, pd, u64, dbl, dbl, dbl, dbl, u64]
    L.c2b_add_sin_noise.argtypes = [vp, pd, u64, pd, u64, pd, pd, dbl, dbl]
    L.c2b_noise_timing.argtypes = [vp, pf]
    L.c2b_add_drift_resident.argtypes = [vp, dbl, dbl, dbl, pd, u64]
    L.c2b_add_noise_resident.argtypes = [vp, dbl, dbl, dbl, dbl, u64]
    L.c2b_add_sin_noise_resident.argtypes = [vp, pd, pd, dbl, dbl]
    L.c2b_download_problem.argtypes = [vp, pd, pd]
    L.c2b_mean_std.argtypes = [vp, pd, u64, pd, u64, pd, pd]
    L.c2b_cull_problem.argtypes = [vp, pd, u64, pd, u64, C.POINTER(u64), pu32, pd, C.POINTER(CullStats)]
    L.c2b_cull_problem_resident.argtypes = [vp, C.POINTER(CullStats)]
    L.c2b_add_incorrect_correspondences.argtypes = [vp, C.POINTER(u64), u64, pu32, pd, dbl, u64,
                                                    C.POINTER(MismatchStats)]
    L.c2b_add_incorrect_correspondences_resident.argtypes = [vp, dbl, u64, C.POINTER(MismatchStats)]
    L.c2b_write_bal.argtypes = [vp, C.c_char_p, i32, pd, u64, pd, u64, C.POINTER(u64), pu32, pd, C.POINTER(BalStats)]
    L.c2b_write_bal_resident.argtypes = [vp, C.c_char_p, i32, C.POINTER(BalStats)]
    L.c2b_read_bal_resident.argtypes = [vp, C.c_char_p, i32, C.POINTER(BalReadStats)]
    L.c2b_probe_fp64.argtypes = [vp, pd]
    L.c2b_generate_world_points_uniform.argtypes = [vp, pf, u64, pu32, u64, pd, u64, u64, dbl, u64, pd,
                                                    C.POINTER(u64)]
    L.c2b_grid_num_cameras.argtypes = [u64, u64]
    L.c2b_grid_num_cameras.restype = u64
    L.c2b_grid_num_points.argtypes = [u64, u64]
    L.c2b_grid_num_points.restype = u64
    L.c2b_grid_cameras.argtypes = [u64, u64, dbl, dbl, pd]
    L.c2b_grid_points.argtypes = [u64, u64, dbl, dbl, dbl, pd]
    L.c2b_line_cameras.argtypes = [u64, dbl, dbl, pd]
    L.c2b_line_points.argtypes = [u64, dbl, dbl, dbl, pd]
    L.c2b_city_mesh.argtypes = [u64, dbl, dbl, dbl, pf, pu32]
    L.c2b_camera_center.argtypes = [pd, pd]
    L.c2b_camera_center.restype = None
    L.c2b_camera_project_world.argtypes = [pd, pd, pd]
    L.c2b_camera_project_world.restype = None
    L.c2b_camera_project.argtypes = [pd, pd, pd]
    L.c2b_camera_project.restype = None
    L.c2b_camera_from_position_direction.argtypes = [pd, pd, pd]
    L.c2b_camera_from_position_direction.restype = None
    L.c2b_camera_transform.argtypes = [pd, pd, pd, pd]
    L.c2b_camera_transform.restype = None
    L.c2b_camera_to_vec.argtypes = [pd, pd]
    L.c2b_camera_to_vec.restype = None
    L.c2b_camera_from_vec.argtypes = [pd, pd]
    L.c2b_camera_from_vec.restype = None
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise C2BError(rc, lib().c2b_last_error().decode("utf-8", "replace"))


class Context:
    """One c2b_ctx = one GPU.  Raises C2BError(-2) when no sm_100 device is visible."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        check(lib().c2b_init(int(device), C.byref(self._h)))
        self.device = int(device)

    @property
    def handle(self):
        return self._h

    def tune(self, name: str, value: float):
        """measurement / test hook (include/city2ba_cuda.h: c2b_tune); name "reset" restores the defaults"""
        check(lib().c2b_tune(self._h, name.encode(), float(value)))

    def close(self):
        if self._h:
            lib().c2b_shutdown(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiContext:
    """c2b_multi: one process driving n GPUs of one box (camera ranges, one NCCL communicator)."""

    def __init__(self, n_gpus: int, devices=None):
        self._h = C.c_void_p()
        dev = (C.c_int * n_gpus)(*devices) if devices is not None else None
        check(lib().c2b_init_multi(int(n_gpus), dev, C.byref(self._h)))
        self.n_gpus = int(n_gpus)

    @property
    def handle(self):
        return self._h

    def tune(self, name: str, value: float):
        for g in range(self.n_gpus):
            check(lib().c2b_tune(lib().c2b_multi_ctx(self._h, g), name.encode(), float(value)))

    def close(self):
        if self._h:
            lib().c2b_shutdown_multi(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx = {}


def context(device: int | None = None) -> Context:
    """Process-wide context for `device` (default: LOCAL_RANK, else 0)."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]
