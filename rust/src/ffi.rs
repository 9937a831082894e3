// Raw bindings to include/city2ba_cuda.h (ABI version 3): EVERY exported symbol, in the header's order
// (tests/test_abi.py::test_rust_ffi_declares_every_export keeps the two lists equal).  NOT compiled in this
// image (no rustc/cargo); the same ABI is exercised end to end by city2ba_b200/_lib.py (ctypes) and by the C++
// host mirror (include/city2ba.hpp) in tests/.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_double, c_float, c_int};

pub const C2B_ABI_VERSION: c_int = 3;
pub const C2B_MAX_GPUS: usize = 16;

#[repr(C)] pub struct c2b_ctx { _p: [u8; 0] }
#[repr(C)] pub struct c2b_scene { _p: [u8; 0] }
#[repr(C)] pub struct c2b_multi { _p: [u8; 0] }
#[repr(C)] pub struct c2b_multi_scene { _p: [u8; 0] }

#[repr(C)] #[derive(Clone, Copy)]
pub struct c2b_vis_options {
    pub cull_mode: c_int, pub occlusion: c_int, pub endpoint_guard_rel: c_int,
    pub count_traversal: c_int, pub block_length: c_double, pub block_inset: c_double,
    pub predicate: c_int, pub reserved: c_int,
}

#[repr(C)]
pub struct c2b_obs {
    pub n_cameras: u64, pub n_obs: u64,
    pub offsets: *mut u64, pub point_idx: *mut u32, pub uv: *mut c_double,
    pub n_candidates: u64, pub pairs_evaluated: u64, pub nodes_visited: u64, pub tris_tested: u64,
    pub h2d_bytes: u64, pub d2h_bytes: u64,
    pub ms_h2d: c_float, pub ms_prep: c_float, pub ms_cull: c_float, pub ms_sort: c_float,
    pub ms_traverse: c_float, pub ms_compact: c_float, pub ms_d2h: c_float, pub ms_total: c_float,
}

#[repr(C)]
pub struct c2b_multi_stats {
    pub n_gpus: c_int,
    pub cam_begin: [u64; C2B_MAX_GPUS], pub cam_end: [u64; C2B_MAX_GPUS],
    pub n_obs: [u64; C2B_MAX_GPUS], pub obs_base: [u64; C2B_MAX_GPUS],
    pub ms_points: [c_float; C2B_MAX_GPUS], pub ms_compute: [c_float; C2B_MAX_GPUS],
    pub ms_exchange: [c_float; C2B_MAX_GPUS], pub ms_d2h: [c_float; C2B_MAX_GPUS],
    pub ms_wall: c_float,
}

// BAProblem::cull on the GPU (c2b_cull_problem / c2b_cull_problem_resident)
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct c2b_cull_stats {
    pub n_cameras: u64, pub n_points: u64, pub n_obs: u64,
    pub iterations: u32, pub reserved: u32,
    pub ms_h2d: c_float, pub ms_compute: c_float, pub ms_d2h: c_float,
}

// noise::add_incorrect_correspondences on the GPU (c2b_add_incorrect_correspondences[_resident])
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct c2b_mismatch_stats {
    pub n_selected: u64, pub n_swapped: u64,
    pub ms_h2d: c_float, pub ms_compute: c_float, pub ms_d2h: c_float,
}

// noise::join_landmarks on the GPU (c2b_join_landmarks[_resident])
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct c2b_join_stats {
    pub n_selected: u64, pub n_changed: u64,
    pub ms_h2d: c_float, pub ms_compute: c_float, pub ms_d2h: c_float,
}

// BAL files on the GPU (c2b_write_bal / c2b_write_bal_resident)
pub const C2B_BAL_TEXT: c_int = 0;
pub const C2B_BAL_BINARY: c_int = 1;
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct c2b_bal_stats {
    pub bytes: u64, pub chunks: u64,
    pub ms_encode: c_float, pub ms_d2h: c_float, pub ms_write: c_float,
}

// BAL files read on the GPU into the resident problem (c2b_read_bal_resident)
pub const C2B_ERR_PARSE: c_int = -8;
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct c2b_bal_read_stats {
    pub n_cameras: u64, pub n_points: u64, pub n_obs: u64,
    pub bytes: u64, pub chunks: u64, pub slow_tokens: u64,
    pub regrouped: u32, pub reserved: u32,
    pub ms_read: c_float, pub ms_h2d: c_float, pub ms_parse: c_float,
}

// Embree's RTCRay layout (48 bytes): what embree_rs::Ray wraps (src/generate.rs:253-262, :457-464)
#[repr(C)] #[derive(Clone, Copy)]
pub struct c2b_ray48 {
    pub org_x: c_float, pub org_y: c_float, pub org_z: c_float, pub tnear: c_float,
    pub dir_x: c_float, pub dir_y: c_float, pub dir_z: c_float, pub time: c_float,
    pub tfar: c_float, pub mask: u32, pub id: u32, pub flags: u32,
}

extern "C" {
    // ---- lifetime ----
    pub fn c2b_init(device: c_int, out: *mut *mut c2b_ctx) -> c_int;
    pub fn c2b_shutdown(ctx: *mut c2b_ctx);
    pub fn c2b_last_error() -> *const c_char;
    pub fn c2b_abi_version() -> c_int;
    pub fn c2b_kernel_launches() -> u64;
    pub fn c2b_tune(ctx: *mut c2b_ctx, name: *const c_char, value: c_double) -> c_int;
    pub fn c2b_probe_fp64(ctx: *mut c2b_ctx, dfma_per_s: *mut c_double) -> c_int;
    // ---- scene ----
    pub fn c2b_scene_create(ctx: *mut c2b_ctx, xyz: *const c_float, nv: u64,
                            tri: *const u32, nt: u64, out: *mut *mut c2b_scene) -> c_int;
    pub fn c2b_scene_bounds(s: *const c2b_scene, lo: *mut c_float, hi: *mut c_float) -> c_int;
    pub fn c2b_scene_num_triangles(s: *const c2b_scene) -> u64;
    pub fn c2b_scene_num_nodes(s: *const c2b_scene) -> u64;
    pub fn c2b_scene_destroy(s: *mut c2b_scene);
    // ---- ray-level entries: any-hit batch (occluded_stream_aos): tfar = -inf on a hit; closest hit of a
    // batch (generate_cameras_poisson's downward rays in one launch): flags = 1 and tfar = distance ----
    pub fn c2b_occluded(ctx: *mut c2b_ctx, s: *const c2b_scene, rays: *mut c2b_ray48, n: u64) -> c_int;
    pub fn c2b_intersect(ctx: *mut c2b_ctx, s: *const c2b_scene, rays: *mut c2b_ray48, n: u64) -> c_int;
    pub fn c2b_intersect1(ctx: *mut c2b_ctx, s: *const c2b_scene, org: *const c_float,
                          dir: *const c_float, hit: *mut c_int, tfar: *mut c_float) -> c_int;
    // ---- the hot path ----
    pub fn c2b_vis_options_default(opt: *mut c2b_vis_options);
    pub fn c2b_visibility_graph(ctx: *mut c2b_ctx, s: *const c2b_scene, cams: *const c_double,
                                c: u64, pts: *const c_double, p: u64, max_dist: c_double,
                                opt: *const c2b_vis_options, out: *mut c2b_obs) -> c_int;
    pub fn c2b_obs_free(ctx: *mut c2b_ctx, obs: *mut c2b_obs);
    pub fn c2b_upload_points(ctx: *mut c2b_ctx, pts: *const c_double, p: u64) -> c_int;
    pub fn c2b_upload_points_device(ctx: *mut c2b_ctx, d_pts: *const c_double, p: u64) -> c_int;
    pub fn c2b_points_device_buffer(ctx: *mut c2b_ctx, capacity: u64, d_out: *mut *mut c_double) -> c_int;
    pub fn c2b_points_commit(ctx: *mut c2b_ctx, p: u64) -> c_int;
    pub fn c2b_upload_cameras(ctx: *mut c2b_ctx, cams: *const c_double, c: u64) -> c_int;
    pub fn c2b_drop_point_grid(ctx: *mut c2b_ctx) -> c_int;
    pub fn c2b_visibility_graph_resident(ctx: *mut c2b_ctx, s: *const c2b_scene, max_dist: c_double,
                                         opt: *const c2b_vis_options, stats_out: *mut c2b_obs) -> c_int;
    pub fn c2b_download_obs(ctx: *mut c2b_ctx, out: *mut c2b_obs) -> c_int;
    pub fn c2b_download_obs_into(ctx: *mut c2b_ctx, obs_base: u64, offsets_dst: *mut u64, idx_dst: *mut u32,
                                 uv_dst: *mut c_double, with_end: c_int, ms_d2h: *mut c_float) -> c_int;
    // ---- several GPUs of one box (rayon's par_iter over cameras, src/generate.rs:434-441, 479-481) ----
    pub fn c2b_init_multi(n_gpus: c_int, devices: *const c_int, out: *mut *mut c2b_multi) -> c_int;
    pub fn c2b_shutdown_multi(m: *mut c2b_multi);
    pub fn c2b_multi_num_gpus(m: *const c2b_multi) -> c_int;
    pub fn c2b_multi_ctx(m: *mut c2b_multi, g: c_int) -> *mut c2b_ctx;
    pub fn c2b_scene_create_multi(m: *mut c2b_multi, xyz: *const c_float, nv: u64, tri: *const u32, nt: u64,
                                  out: *mut *mut c2b_multi_scene) -> c_int;
    pub fn c2b_scene_destroy_multi(s: *mut c2b_multi_scene);
    pub fn c2b_multi_scene_get(s: *const c2b_multi_scene, g: c_int) -> *mut c2b_scene;
    pub fn c2b_visibility_graph_multi(m: *mut c2b_multi, s: *const c2b_multi_scene, cams: *const c_double, c: u64,
                                      pts: *const c_double, p: u64, max_dist: c_double,
                                      opt: *const c2b_vis_options, out: *mut c2b_obs,
                                      stats: *mut c2b_multi_stats) -> c_int;
    pub fn c2b_reprojection_error_resident(ctx: *mut c2b_ctx, norm: c_double, out: *mut c_double) -> c_int;
    // ---- noise pass (src/noise.rs:35-177, 388-416) ----
    pub fn c2b_add_drift(ctx: *mut c2b_ctx, cams: *mut c_double, c: u64, pts: *mut c_double, p: u64,
                         strength: c_double, angle_strength: c_double, std: c_double,
                         dir: *const c_double, seed: u64) -> c_int;
    pub fn c2b_add_drift_normalized(ctx: *mut c2b_ctx, cams: *mut c_double, c: u64, pts: *mut c_double, p: u64,
                                    strength: c_double, angle_strength: c_double, std: c_double, seed: u64) -> c_int;
    pub fn c2b_add_noise(ctx: *mut c2b_ctx, cams: *mut c_double, c: u64, pts: *mut c_double, p: u64,
                         uv: *mut c_double, o: u64, translation_std: c_double, rotation_std: c_double,
                         point_std: c_double, observations_std: c_double, seed: u64) -> c_int;
    pub fn c2b_add_sin_noise(ctx: *mut c2b_ctx, cams: *mut c_double, c: u64, pts: *mut c_double, p: u64,
                             dir: *const c_double, noise_dir: *const c_double, strength: c_double,
                             frequency: c_double) -> c_int;
    pub fn c2b_add_drift_resident(ctx: *mut c2b_ctx, strength: c_double, angle_strength: c_double, std: c_double,
                                  dir: *const c_double, seed: u64) -> c_int;
    pub fn c2b_add_noise_resident(ctx: *mut c2b_ctx, translation_std: c_double, rotation_std: c_double,
                                  point_std: c_double, observations_std: c_double, seed: u64) -> c_int;
    pub fn c2b_add_sin_noise_resident(ctx: *mut c2b_ctx, dir: *const c_double, noise_dir: *const c_double,
                                      strength: c_double, frequency: c_double) -> c_int;
    pub fn c2b_download_problem(ctx: *mut c2b_ctx, cams_out: *mut c_double, pts_out: *mut c_double) -> c_int;
    pub fn c2b_noise_timing(ctx: *mut c2b_ctx, ms: *mut c_float) -> c_int;
    pub fn c2b_mean_std(ctx: *mut c2b_ctx, cams: *const c_double, c: u64, pts: *const c_double, p: u64,
                        mean: *mut c_double, std: *mut c_double) -> c_int;
    // ---- graph post-processing: a Rust BAProblem::cull would call c2b_cull_problem (INTEGRATION.md) ----
    pub fn c2b_cull_problem(ctx: *mut c2b_ctx, cams: *mut c_double, c: u64, pts: *mut c_double, p: u64,
                            offsets: *mut u64, point_idx: *mut u32, uv: *mut c_double,
                            out: *mut c2b_cull_stats) -> c_int;
    pub fn c2b_cull_problem_resident(ctx: *mut c2b_ctx, out: *mut c2b_cull_stats) -> c_int;
    pub fn c2b_add_incorrect_correspondences(ctx: *mut c2b_ctx, offsets: *const u64, c: u64, point_idx: *mut u32,
                                             uv: *const c_double, mismatch_chance: c_double, seed: u64,
                                             out: *mut c2b_mismatch_stats) -> c_int;
    pub fn c2b_add_incorrect_correspondences_resident(ctx: *mut c2b_ctx, mismatch_chance: c_double, seed: u64,
                                                      out: *mut c2b_mismatch_stats) -> c_int;
    pub fn c2b_join_landmarks(ctx: *mut c2b_ctx, pts: *const c_double, p: u64, offsets: *const u64, c: u64,
                              point_idx: *mut u32, join_percent: c_double, seed: u64,
                              out: *mut c2b_join_stats) -> c_int;
    pub fn c2b_join_landmarks_resident(ctx: *mut c2b_ctx, join_percent: c_double, seed: u64,
                                       out: *mut c2b_join_stats) -> c_int;
    // ---- BAL files: a Rust BAProblem::write would call c2b_write_bal with the format of its extension ----
    pub fn c2b_write_bal(ctx: *mut c2b_ctx, path: *const c_char, format: c_int, cams: *const c_double, c: u64,
                         pts: *const c_double, p: u64, offsets: *const u64, point_idx: *const u32,
                         uv: *const c_double, out: *mut c2b_bal_stats) -> c_int;
    pub fn c2b_write_bal_resident(ctx: *mut c2b_ctx, path: *const c_char, format: c_int,
                                  out: *mut c2b_bal_stats) -> c_int;
    pub fn c2b_read_bal_resident(ctx: *mut c2b_ctx, path: *const c_char, format: c_int,
                                 out: *mut c2b_bal_read_stats) -> c_int;
    // ---- input generation ----
    pub fn c2b_generate_world_points_uniform(ctx: *mut c2b_ctx, xyz: *const c_float, nv: u64, tri: *const u32,
                                             nt: u64, cams: *const c_double, c: u64, num_points: u64,
                                             max_dist: c_double, seed: u64, pts_out: *mut c_double,
                                             n_out: *mut u64) -> c_int;
    // host-side generators (the Rust crate has its own synthetic.rs; bound for tests / tools)
    pub fn c2b_grid_num_cameras(cameras_per_block: u64, num_blocks: u64) -> u64;
    pub fn c2b_grid_num_points(points_per_block: u64, num_blocks: u64) -> u64;
    pub fn c2b_grid_cameras(cameras_per_block: u64, num_blocks: u64, block_length: c_double,
                            camera_height: c_double, cams_out: *mut c_double) -> c_int;
    pub fn c2b_grid_points(points_per_block: u64, num_blocks: u64, block_length: c_double, block_inset: c_double,
                           point_height: c_double, pts_out: *mut c_double) -> c_int;
    pub fn c2b_line_cameras(num_cameras: u64, length: c_double, camera_height: c_double, cams_out: *mut c_double) -> c_int;
    pub fn c2b_line_points(num_points: u64, length: c_double, point_offset: c_double, point_height: c_double,
                           pts_out: *mut c_double) -> c_int;
    pub fn c2b_city_mesh(num_blocks: u64, block_length: c_double, block_inset: c_double, height: c_double,
                         xyz_out: *mut c_float, tri_out: *mut u32) -> c_int;
    pub fn c2b_camera_center(cam: *const c_double, out: *mut c_double);
    pub fn c2b_camera_project_world(cam: *const c_double, p: *const c_double, out: *mut c_double);
    pub fn c2b_camera_project(cam: *const c_double, pc: *const c_double, out: *mut c_double);
    pub fn c2b_camera_from_position_direction(pos: *const c_double, r: *const c_double, cam_out: *mut c_double);
    pub fn c2b_camera_transform(cam: *const c_double, d_r: *const c_double, dloc: *const c_double,
                                cam_out: *mut c_double);
    pub fn c2b_camera_to_vec(cam: *const c_double, out: *mut c_double);
    pub fn c2b_camera_from_vec(v: *const c_double, cam_out: *mut c_double);
}
