#!/usr/bin/env python
"""bench.py — camera x point visibility tests/s on a synthetic city grid (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg3|cfg4|cfg5]
                    [--cull-mode grid|exhaustive] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path (c2b_visibility_graph: point grid -> plan -> fused cull + occlusion ->
sort + write) over the whole workload; cameras are sharded across GPUs (contiguous ranges, the mesh, BVH and
points replicated), so total work is fixed as N grows ("strong" scaling on the named configuration).  Prints
ONE JSON line on rank 0.

  value : C*P / t with inputs resident in HBM, t = device time of the step (CUDA events on the library's
          stream), max over ranks.  The point grid is derived data (it depends on max_dist), so it is dropped
          before every timed step and its build is inside t; `value_cached_grid` is the same with the grid
          kept between calls.
  e2e   : the same metric through the host-buffer C-ABI call, wall clock around the call: pinned host inputs
          copied H2D and the CSR result copied D2H inside the timed region.  N = 1: c2b_visibility_graph.
          N > 1: rank 0 drives all N GPUs through the library's own multi-GPU entry
          (c2b_visibility_graph_multi: per-GPU point shards + NCCL all-gather, one NCCL all-gather of the
          per-GPU counts, every GPU writes its slab into ONE pinned host CSR); the clock stops when that CSR
          is complete.  `e2e_pageable`: the same with pageable (numpy) inputs; `e2e_cold`: first call on a
          fresh ctx (every device and pinned buffer allocated inside the call).
  parity: rows of an evenly spaced camera sample of the e2e result compared bit for bit with the oracle's CPU
          arm (the cpu_baseline sample at N = 1); result_hash: order-sensitive 64-bit hash of the whole CSR,
          independent of N, checked against tests/golden/result_hashes.json.
  --impl reference : the reference's algorithm on the box's host cores (the oracle's OpenMP + CPU-BVH arm,
          built -O3 -march=native on the box; the Rust/Embree reference cannot be built in this image), on a
          bounded camera sample of the same workload.
  --dump-outputs DIR : after the run, the CSR the e2e call returned in its last timed step as float64 .npy files
          (see dump_outputs), so that two builds can be compared output for output on the same inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the checkout may be read-only: the bench writes nothing into it

WORKLOADS = {
    # name: (blocks, cameras_per_block, points_per_block)  — BASELINE.md section 4
    "cfg2": (4, 10, 10),
    "cfg3": (16, 9, 306),
    "cfg4": (64, 6, 200),
    # config 5: the same 64x64 city with every wall tessellated 11 x 11 and displaced (4.96 M triangles),
    # 49,920 lattice cameras, 4,992,000 points sampled on the mesh (area-weighted, seeded)
    "cfg5": (64, 3, 100),
    "cfg5s": (16, 3, 100),  # a 16x16-block cut of cfg5 (310 k triangles) for quick runs
}
TESS_K = 11
MAX_DIST = 10.0
BLOCK_LENGTH, BLOCK_INSET, CAM_H, PT_H, BUILDING_H = 20.0, 1.0, 1.0, 1.0, 10.0
HASHES = os.path.join(ROOT, "tests", "golden", "result_hashes.json")


def trace(msg):
    """progress on stderr when C2B_BENCH_TRACE=1 (debugging multi-rank runs)"""
    if os.environ.get("C2B_BENCH_TRACE") == "1":
        print(f"[bench rank {os.environ.get('RANK', '0')} {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def ncu_traffic(stage, workload, cull_mode):
    """dram__bytes_read.sum + dram__bytes_write.sum of the stage's kernel, per launch, from the
    committed `ncu --set full` capture (profiles/traffic.json, written by profiles/summarize.py);
    None when no capture matches this workload."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(p))
        e = t[f"{workload}/{cull_mode}/{stage}"]
        return float(e["dram_bytes"]), f'{e["kernel"]}: {e["source"]}'
    except Exception:
        return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(
                ["nvidia-smi", "-i", str(device), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        time.sleep(0.25)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for k, nm in enumerate(names):
                    if r[3 + k].strip().lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)),
                   "reasons": sorted(reasons), "samples": len(sm)}
        return out


def city_mesh_tessellated(n, k):
    # plain numpy (no library call): city2ba_b200.synthetic imports without mapping the CUDA library
    from city2ba_b200.synthetic import city_mesh_tessellated as f
    return f(n, k, BLOCK_LENGTH, BLOCK_INSET, BUILDING_H)


def build_workload(name, gen="product"):
    """(cameras, points, xyz, tri) of a BASELINE config.  gen = "product": the library's host generators
    (c2b_grid_*); gen = "oracle": the oracle's own (the reference arm never maps the CUDA library; the two
    are checked equal in tests/test_host_mirror.py)."""
    n, cpb, ppb = WORKLOADS[name]
    if gen == "oracle":
        from oracle import oracle as g
        cams = g.grid_cameras(cpb, n, BLOCK_LENGTH, CAM_H)
        lattice = lambda: g.grid_points(ppb, n, BLOCK_LENGTH, BLOCK_INSET, PT_H)  # noqa: E731
        box_mesh = lambda: g.city_mesh(n, BLOCK_LENGTH, BLOCK_INSET, BUILDING_H)  # noqa: E731
    else:
        from city2ba_b200 import synthetic as g
        cams = g.grid_cameras(cpb, n, BLOCK_LENGTH, CAM_H)
        lattice = lambda: g.grid_points(ppb, n, BLOCK_LENGTH, BLOCK_INSET, PT_H)  # noqa: E731
        box_mesh = lambda: g.city_mesh(n, BLOCK_LENGTH, BLOCK_INSET, BUILDING_H)  # noqa: E731
    if name.startswith("cfg5"):
        xyz, tri = city_mesh_tessellated(n, TESS_K)
        pts = sample_points_on_walls(xyz, tri, 12 * ppb * n * (n + 1))
        return cams, pts, xyz, tri
    pts = lattice()
    xyz, tri = box_mesh()
    return cams, pts, xyz, tri


def describe(name, C, P):
    n = WORKLOADS[name][0]
    return (f"{name}: synthetic {n}x{n}-block city{', walls tessellated' if name.startswith('cfg5') else ''}, "
            f"{C} cameras x {P} points, max_dist {MAX_DIST}")


def sample_points_on_walls(xyz, tri, n, seed=0xC17B2A):
    """n world points on the mesh, area-weighted over the triangles that reach below 3 m (what
    street-level cameras can see), uniform inside each triangle — the rule of src/generate.rs:370-408 with a
    seeded generator (the reference's thread_rng cannot be seeded)."""
    rng = np.random.default_rng(seed)
    a, b, c = (xyz[tri[:, k]].astype(np.float64) for k in range(3))
    low = np.minimum(np.minimum(a[:, 1], b[:, 1]), c[:, 1]) <= 3.0
    a, b, c = a[low], b[low], c[low]
    area = 0.5 * np.linalg.norm(np.cross(b - a, c - a), axis=1)
    cdf = np.cumsum(area)
    pick = np.minimum(np.searchsorted(cdf, rng.uniform(0, cdf[-1], n)), len(cdf) - 1)
    r1, r2 = rng.uniform(size=n), rng.uniform(size=n)
    flip = r1 + r2 > 1
    r1[flip], r2[flip] = 1 - r1[flip], 1 - r2[flip]
    return np.ascontiguousarray(a[pick] + r1[:, None] * (b[pick] - a[pick]) + r2[:, None] * (c[pick] - a[pick]))


def shard(C, rank, world):
    return (rank * C) // world, ((rank + 1) * C) // world


# ---- result hash: order-sensitive inside a camera, additive over cameras (so it does not depend on how
# the cameras were split over GPUs) ------------------------------------------------------------------------
_K = [np.uint64(k) for k in (0x9E3779B97F4A7C15, 0xBF58476D1CE4E5B9, 0x94D049BB133111EB, 0xD6E8FEB86659FD93,
                             0xA0761D6478BD642F, 0xE7037ED1A0B428DB)]


def result_hash(offsets, idx, uv, cam0=0, chunk=8192) -> int:
    """64-bit hash of a CSR slab whose first camera has global index cam0: per observation a mix of (point
    index, u bits, v bits, position in the row); per camera the wrapped sum of those, mixed with the camera's
    global index and its count; the wrapped sum over cameras."""
    off = np.asarray(offsets, np.int64)
    idx = np.asarray(idx)
    uvb = np.ascontiguousarray(uv, np.float64).reshape(-1).view(np.uint64).reshape(-1, 2)
    C = len(off) - 1
    total = np.uint64(0)
    with np.errstate(over="ignore"):
        for a in range(0, C, chunk):
            b = min(C, a + chunk)
            o0, o1 = int(off[a]), int(off[b])
            n = (off[a + 1:b + 1] - off[a:b]).astype(np.uint64)
            cam = (np.arange(a, b, dtype=np.uint64) + np.uint64(cam0))
            s = np.zeros(b - a, np.uint64)
            if o1 > o0:
                pos = (np.arange(o0, o1, dtype=np.int64) - np.repeat(off[a:b], n.astype(np.int64))).astype(np.uint64)
                h = (idx[o0:o1].astype(np.uint64) + np.uint64(1)) * _K[0]
                h ^= uvb[o0:o1, 0] * _K[1]
                h ^= uvb[o0:o1, 1] * _K[2]
                h ^= (pos + np.uint64(1)) * _K[3]
                h ^= h >> np.uint64(29)
                h *= _K[4]
                h ^= h >> np.uint64(32)
                nz = n > 0
                s[nz] = np.add.reduceat(h, (off[a:b][nz] - o0))
            g = (s + n * _K[5]) * (np.uint64(2) * cam + np.uint64(1))
            g ^= g >> np.uint64(31)
            total = total + g.sum(dtype=np.uint64)
    return int(total)


def expected_hash(workload):
    try:
        return int(json.load(open(HASHES))[workload], 16)
    except Exception:
        return None


DUMP_MAX_OBS = 2_000_000  # 48 MB of (point index, u, v) in float64; with the offsets under 64 MB at every workload


def dump_outputs(out_dir, offsets, idx, uv, seed=0):
    """Writes a CSR (offsets, idx, uv) as float64 arrays (exact: indices and offsets are below 2**53):
    offsets.npy, all C + 1 entries; point_idx.npy (O,) and uv.npy (O, 2), every observation, or, when there are
    more than DUMP_MAX_OBS (cfg4: 53 M), the observations at a seeded sample of positions, ascending, which is
    the same sample for two results with the same number of observations."""
    O = len(idx)
    sel = slice(None) if O <= DUMP_MAX_OBS else np.unique(np.random.default_rng(seed).integers(0, O, DUMP_MAX_OBS))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "offsets.npy"), np.asarray(offsets, np.float64))
    np.save(os.path.join(out_dir, "point_idx.npy"), np.asarray(idx)[sel].astype(np.float64))
    np.save(os.path.join(out_dir, "uv.npy"), np.asarray(uv, np.float64).reshape(-1, 2)[sel])


def parity_against(sample_idx, vis, offsets, idx, uv):
    """rows `sample_idx` of the CSR (offsets, idx, uv) against the oracle graph `vis` of those cameras"""
    off = np.asarray(offsets, np.int64)
    rn = np.diff(vis.offsets.astype(np.int64))
    n = off[sample_idx + 1] - off[sample_idx]
    bad = n != rn
    uv2 = np.asarray(uv).reshape(-1, 2)
    for k in np.nonzero(~bad)[0]:
        a, b = off[sample_idx[k]], off[sample_idx[k] + 1]
        ra, rb = int(vis.offsets[k]), int(vis.offsets[k + 1])
        # (u, v) compared as raw 64-bit words: the sign of a zero counts (v = +-0 all over the synthetic cities)
        same_uv = np.array_equal(np.ascontiguousarray(uv2[a:b], np.float64).view(np.uint64),
                                 np.ascontiguousarray(vis.uv[ra:rb], np.float64).view(np.uint64))
        if not (np.array_equal(np.asarray(idx[a:b], np.uint64), vis.point_idx[ra:rb]) and same_uv):
            bad[k] = True
    return {"cameras_checked": int(len(sample_idx)), "observations_checked": int(rn.sum()),
            "mismatches": int(bad.sum()), "against": "oracle CPU arm (orc_ref_visibility_graph), bit for bit: "
            "row lengths, point indices, (u, v)"}


def cpu_arm(cams, pts, xyz, tri, budget_s, threads=0, fixed_n=None):
    """Times the oracle's multithreaded CPU arm on a bounded camera sample (every k-th camera).
    Returns (tests_per_s, cores, sample description, obs_per_s, sample camera indices, sample graph)."""
    from oracle import oracle as orc
    C, P = len(cams), len(pts)
    ncores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    if threads <= 0:
        threads = ncores  # explicit: torchrun exports OMP_NUM_THREADS=1, which would serialise the arm
    n = min(C, fixed_n if fixed_n else max(ncores, 8))
    for _ in range(4):  # grow the sample until it fills about the budget
        idx = np.unique(np.linspace(0, C - 1, n).astype(np.int64))
        t0 = time.perf_counter()
        v, used = orc.ref_visibility_graph(xyz, tri, cams[idx], pts, MAX_DIST, n_threads=threads)
        dt = time.perf_counter() - t0
        if fixed_n or dt >= 0.5 * budget_s or n >= C:
            break
        n = int(min(C, max(n + used, 0.9 * n * budget_s / max(dt, 1e-6))))
        n = max(used, (n // used) * used)
    return (len(idx) * P / dt, used, f"{len(idx)} of {C} cameras (evenly spaced) x all {P} points, {dt:.1f} s",
            v.n_obs / dt, idx, v)


def run_reference(args):
    """--impl reference: the CPU arm, rank 0 only.  Inputs from the oracle's own generators: this process
    never maps libcity2ba_cuda.so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ["C2B_ORACLE_NATIVE"] = "1"
    cams, pts, xyz, tri = build_workload(args.workload, gen="oracle")
    C, P = len(cams), len(pts)
    budget = 8.0
    vals, obs = [], []
    cores, sample = 1, ""
    for s in range(args.warmup + args.steps):
        v, cores, sample, o, _, _ = cpu_arm(cams, pts, xyz, tri, budget)
        if s >= args.warmup:
            vals.append(v)
            obs.append(o)
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": "camera-point visibility tests/sec", "value": value,
        "unit": "tests/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * C * P / value, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": describe(args.workload, C, P), "cameras": C, "points": P,
                   "triangles": int(len(tri)), "note": "reference binary (Rust + Embree 3.8) cannot be "
                   "built here; this is the oracle's C restatement of its algorithm: OpenMP over "
                   "cameras, brute-force point loop, CPU BVH any-hit, compiled -O3 -march=native on this box; "
                   "ms_per_step extrapolates the sample to the whole workload"},
        "observations_per_s": float(np.mean(obs)),
        "cpu_baseline": {"value": value, "unit": "tests/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "tests/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--cull-mode", default="grid", choices=["grid", "exhaustive"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-exhaustive", action="store_true")
    ap.add_argument("--no-noise", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the cfg3 / cfg5 lines of the default run")
    ap.add_argument("--no-extras", action="store_true", help="skip e2e_pageable / e2e_cold")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the CSR of the last timed e2e step to DIR/{offsets,point_idx,uv}.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU result; --impl reference computes a camera sample only")
    default_run = args.workload is None
    if args.workload is None:
        # the metric's target is quoted on the 64x64-block city (cfg4); it fits one GPU
        args.workload = "cfg4"
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    os.environ["C2B_ORACLE_NATIVE"] = "1"  # the CPU arm below is built -O3 -march=native on this box
    # stdout carries exactly ONE JSON line: anything a library prints there (NCCL announces its version on
    # stdout when a communicator is created) goes to stderr instead; the line is written to the saved descriptor
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    import ctypes as Ct

    import torch
    import torch.distributed as dist
    import city2ba_b200 as c2b
    from city2ba_b200 import _lib
    from city2ba_b200.generate import ResidentProblem, _options

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        cpu_group = dist.new_group(backend="gloo")  # host-side waits that must not occupy a GPU
    else:
        torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    ctx = c2b.context(local)
    L = _lib.lib()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    K = args.steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def flush_l2():
        flush.zero_()
        torch.cuda.synchronize()

    def rmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def rsum(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    STAGES = ("ms_total", "ms_prep", "ms_cull", "ms_sort", "ms_traverse", "ms_compact")

    class Problem:
        """one workload on this rank: pinned host copies, the scene, the resident problem"""

        def __init__(self, name):
            self.name = name
            self.cams, self.pts, self.xyz, self.tri = build_workload(name)
            self.C, self.P = len(self.cams), len(self.pts)
            self.c0, self.c1 = shard(self.C, rank, world)
            self.pin_cams = torch.from_numpy(np.ascontiguousarray(self.cams)).pin_memory()
            self.pin_pts = torch.from_numpy(self.pts).pin_memory()
            t0 = time.perf_counter()
            self.scene = c2b.Scene(self.xyz, self.tri, ctx=ctx)
            self.scene_build_ms = 1e3 * (time.perf_counter() - t0)
            self.rp = ResidentProblem(ctx)
            self.opt = _options(args.cull_mode, "mesh", False, False, BLOCK_LENGTH, BLOCK_INSET)

        def upload(self):
            self.rp.upload_points_ptr(self.pin_pts.data_ptr(), self.P)
            self.rp.upload_cameras_ptr(self.pin_cams.data_ptr() + 120 * self.c0, self.c1 - self.c0)
            torch.cuda.synchronize()

        def resident(self, mode, steps, warmup, count=False, drop_grid=True):
            """device-resident arm: (sum of stage ms over the timed steps, stats of the last step)"""
            self.upload()
            st = None
            tot = {k: 0.0 for k in STAGES}
            for s in range(warmup + steps):
                if s == warmup:
                    barrier()
                flush_l2()
                if drop_grid:
                    _lib.check(L.c2b_drop_point_grid(ctx.handle))
                st = self.rp.run(self.scene, MAX_DIST, cull_mode=mode, count_traversal=count)
                if s >= warmup:
                    for k in tot:
                        tot[k] += st[k]
            barrier()
            return tot, st

        def e2e_single(self, steps, warmup, cams_ptr, pts_ptr, the_ctx=None):
            """host buffers -> c2b_visibility_graph -> host CSR on this rank's GPU; wall seconds over `steps`"""
            h = (the_ctx or ctx).handle
            out = _lib.Obs()
            t = 0.0
            for s in range(warmup + steps):
                flush_l2()
                t0 = time.perf_counter()
                _lib.check(L.c2b_visibility_graph(h, self.scene.handle, cams_ptr, self.C, pts_ptr, self.P, MAX_DIST,
                                                  Ct.byref(self.opt), Ct.byref(out)))
                dt = time.perf_counter() - t0
                if s >= warmup:
                    t += dt
            return t, out

    trace("building the workload")
    prob = Problem(args.workload)
    C, P = prob.C, prob.P
    trace(f"workload ready: {C} x {P}")

    # ---- device-resident arm ("value") ----------------------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = L.c2b_kernel_launches()
    tot, st = prob.resident(args.cull_mode, K, args.warmup)
    launches = L.c2b_kernel_launches() - launches0
    launches_per_step = launches // (K + args.warmup)
    t_dev = tot["ms_total"] / 1e3
    tot_cached, _ = prob.resident(args.cull_mode, K, 1, drop_grid=False)
    trace("resident arms done")

    # ---- end-to-end arm: host buffers -> C-ABI call -> ONE host CSR ------------------------------------------
    mctx = mscene = None
    multi_stats = None
    if world == 1:
        e2e_t, out = prob.e2e_single(K, args.warmup, prob.pin_cams.data_ptr(), prob.pin_pts.data_ptr())
    else:
        out = _lib.Obs()
        e2e_t = 0.0
        barrier()
        if rank == 0:
            # the library's multi-GPU entry: this process drives all `world` GPUs (the other ranks wait at the
            # barrier below with their GPUs idle)
            trace("creating the multi-GPU context")
            mctx = c2b.MultiContext(world)
            mscene = c2b.MultiScene(prob.xyz, prob.tri, mctx)
            trace("multi-GPU context and scene ready")
            ms = _lib.MultiStats()
            for s in range(args.warmup + K):
                flush_l2()
                t0 = time.perf_counter()
                _lib.check(L.c2b_visibility_graph_multi(mctx.handle, mscene.handle, prob.pin_cams.data_ptr(), C,
                                                        prob.pin_pts.data_ptr(), P, MAX_DIST, Ct.byref(prob.opt),
                                                        Ct.byref(out), Ct.byref(ms)))
                dt = time.perf_counter() - t0
                if s >= args.warmup:
                    e2e_t += dt
            multi_stats = {k: [round(float(getattr(ms, k)[g]), 4) for g in range(world)]
                           for k in ("ms_points", "ms_compute", "ms_exchange", "ms_d2h")}
            multi_stats["n_obs"] = [int(ms.n_obs[g]) for g in range(world)]
            multi_stats["ms_wall_last_step"] = float(ms.ms_wall)
        # a CPU barrier: an NCCL one would park a spinning kernel on GPUs 1..N-1 while rank 0 is timing them
        trace("e2e arm done, waiting at the host barrier")
        dist.barrier(group=cpu_group)
    clocks = sampler.stop() if sampler else None
    trace("past the e2e arm")

    csr = None
    res_hash = None
    if rank == 0:
        O = int(out.n_obs)
        csr = (np.ctypeslib.as_array(out.offsets, shape=(C + 1,)).copy(),
               np.ctypeslib.as_array(out.point_idx, shape=(max(O, 1),))[:O].copy(),
               np.ctypeslib.as_array(out.uv, shape=(max(2 * O, 1),))[:2 * O].copy())
        res_hash = result_hash(*csr)
    h2d, d2h = int(out.h2d_bytes), int(out.d2h_bytes)
    n_obs_e2e = int(out.n_obs)
    e2e_stage = {k: float(getattr(out, k)) for k in ("ms_h2d", "ms_prep", "ms_cull", "ms_sort", "ms_traverse", "ms_compact", "ms_d2h")}

    # ---- e2e with pageable inputs, and the first call on a fresh ctx (rank 0) ---------------------------------
    extras = {}
    if rank == 0 and not args.no_extras:
        pg_cams, pg_pts = np.array(prob.cams, copy=True), np.array(prob.pts, copy=True)  # plain numpy = pageable
        steps_pg = max(3, K // 2)
        if world == 1:
            t_pg, o2 = prob.e2e_single(steps_pg, 1, pg_cams.ctypes.data, pg_pts.ctypes.data)
            ms_h2d_pg = float(o2.ms_h2d)
            ctx.tune("stage_threads", 0)
            t_drv, o3 = prob.e2e_single(steps_pg, 1, pg_cams.ctypes.data, pg_pts.ctypes.data)
            ctx.tune("reset", 0)
            ms_h2d_drv = float(o3.ms_h2d)
        else:
            o2 = _lib.Obs()
            ms2 = _lib.MultiStats()
            def multi_pageable(n):
                t = 0.0
                for s in range(1 + n):
                    flush_l2()
                    t0 = time.perf_counter()
                    _lib.check(L.c2b_visibility_graph_multi(mctx.handle, mscene.handle, pg_cams.ctypes.data, C,
                                                            pg_pts.ctypes.data, P, MAX_DIST, Ct.byref(prob.opt),
                                                            Ct.byref(o2), Ct.byref(ms2)))
                    if s >= 1:
                        t += time.perf_counter() - t0
                return t
            t_pg = multi_pageable(steps_pg)
            ms_h2d_pg = float(o2.ms_h2d)
            extras["e2e_pageable_per_gpu_last_step"] = {
                k: [round(float(getattr(ms2, k)[g]), 4) for g in range(world)]
                for k in ("ms_points", "ms_compute", "ms_exchange", "ms_d2h")}
            mctx.tune("stage_threads", 0)
            t_drv = multi_pageable(steps_pg)
            mctx.tune("reset", 0)
            ms_h2d_drv = float(o2.ms_h2d)
        extras["e2e_pageable"] = {
            "value": C * P * steps_pg / t_pg, "unit": "tests/s", "ms_per_step": 1e3 * t_pg / steps_pg, "steps": steps_pg,
            "ms_h2d": ms_h2d_pg,
            "driver_staged": {"ms_per_step": 1e3 * t_drv / steps_pg, "ms_h2d": ms_h2d_drv,
                              "note": "stage_threads = 0: cudaMemcpyAsync straight from the pageable arrays"},
            "note": "caller arrays are plain numpy (pageable), what a Rust Vec's as_ptr() is; the library stages "
                    "them through its pinned ring with 4 host threads; results land in the library's pinned CSR"}
        if world == 1:
            cold = _lib.Context(local)
            t0 = time.perf_counter()
            cold_scene = c2b.Scene(prob.xyz, prob.tri, ctx=cold)
            t_scene = time.perf_counter() - t0
            o4 = _lib.Obs()
            t0 = time.perf_counter()
            _lib.check(L.c2b_visibility_graph(cold.handle, cold_scene.handle, pg_cams.ctypes.data, C, pg_pts.ctypes.data, P,
                                              MAX_DIST, Ct.byref(prob.opt), Ct.byref(o4)))
            t_cold = time.perf_counter() - t0
            extras["e2e_cold"] = {
                "value": C * P / t_cold, "unit": "tests/s", "ms": 1e3 * t_cold, "scene_build_ms": 1e3 * t_scene,
                "note": "first call on a fresh c2b_ctx with pageable inputs: every device buffer is allocated inside the "
                        "call and the CSR comes back in unpinned huge-page memory through a pinned ring (pinning 1.1 GB "
                        "would cost 0.55-1.3 s on this host; the second call on a ctx does pin); the CUDA primary "
                        "context already exists"}
            cold_scene.close()
            cold.close()
    if mctx is not None:
        mscene.close()
        mctx.close()
    if world > 1:
        # the other ranks keep their GPUs idle until rank 0 is done driving them (their next arms would time-slice
        # with rank 0's e2e_pageable calls: that cost 11-12 ms per GPU in r02k / r02p)
        dist.barrier(group=cpu_group)

    # ---- noise pass on the generated problem (config 2 / 5: drift + Gaussian noise), N = 1 only ------
    noise = None
    if not args.no_noise and world == 1:
        O = n_obs_e2e
        pd_ = Ct.POINTER(Ct.c_double)
        # pinned host arrays (what a host program that cares about transfer time would hand over)
        t_uv = torch.from_numpy(csr[2].copy() if O else np.zeros(0)).pin_memory()
        t_cam = torch.from_numpy(np.ascontiguousarray(prob.cams).copy()).pin_memory()
        t_pts = torch.from_numpy(prob.pts.copy()).pin_memory()
        uv, ncam, npts = t_uv.numpy(), t_cam.numpy(), t_pts.numpy()
        ms3 = (Ct.c_float * 3)()
        noise = {}
        b_drift = 2 * (120 * C + 24 * P) + 3 * 24 * (C + P)
        b_noise = 2 * (120 * C + 24 * P + 16 * O) + 2 * 24 * (C + P)
        # (1) resident: generate -> noise without leaving HBM; ms_kernels = statistics reductions + elementwise
        # kernels, CUDA events on the library's stream
        prob.upload()
        prob.rp.run(prob.scene, MAX_DIST, cull_mode=args.cull_mode)
        for name, call, nbytes in (
            ("add_drift_normalized", lambda: L.c2b_add_drift_resident(ctx.handle, 0.001, 0.0, 0.0, None, 1), b_drift),
            ("add_noise", lambda: L.c2b_add_noise_resident(ctx.handle, 0.0, 0.0001, 0.01, 0.001, 42), b_noise),
        ):
            kern = 1e9
            for _ in range(4):
                flush_l2()
                _lib.check(call())
                _lib.check(L.c2b_noise_timing(ctx.handle, ms3))
                kern = min(kern, float(ms3[1]))
            noise[name] = {"elements": C + P + (O if name == "add_noise" else 0), "ms_kernels_resident": kern,
                           "algorithmic_bytes": nbytes, "kernel_GBps": nbytes / (kern * 1e-3) / 1e9,
                           "frac_of_hbm_peak": nbytes / (kern * 1e-3) / 1e9 / measured_peaks()[0]}
        # (2) host arrays in and out through the reference-shaped entries
        for name, call in (
            ("add_drift_normalized", lambda: L.c2b_add_drift_normalized(
                ctx.handle, ncam.ctypes.data_as(pd_), len(ncam), npts.ctypes.data_as(pd_), len(npts), 0.001, 0.0, 0.0, 1)),
            ("add_noise", lambda: L.c2b_add_noise(
                ctx.handle, ncam.ctypes.data_as(pd_), len(ncam), npts.ctypes.data_as(pd_), len(npts),
                uv.ctypes.data_as(pd_), O, 0.0, 0.0001, 0.01, 0.001, 42)),
        ):
            best_wall = 1e9
            for _ in range(3):
                t0 = time.perf_counter()
                _lib.check(call())
                best_wall = min(best_wall, time.perf_counter() - t0)
            noise[name]["ms_host_to_host"] = 1e3 * best_wall
            noise[name]["note"] = ("ms_kernels_resident: c2b_add_*_resident on the problem in HBM (statistics + elementwise "
                                   "kernels, CUDA events); ms_host_to_host: pinned host arrays in and out, observations "
                                   "streamed in chunks so that upload and download overlap")

    # ---- traversal counters (one untimed instrumented run) and the exhaustive arm ------------------
    _, stc = prob.resident(args.cull_mode, 1, 0, count=True)
    ex = None
    if not args.no_exhaustive and args.cull_mode == "grid":
        ex_steps = 2 if C * P > 2e11 else 5
        ex_tot, ex_st = prob.resident("exhaustive", ex_steps, 1)
        ex = (ex_tot, ex_st, ex_steps)

    # ---- reduce over ranks (max time, summed work) -----------------------------------------------------
    t_dev_max = rmax(t_dev)
    t_cached_max = rmax(tot_cached["ms_total"] / 1e3)
    e2e_max = rmax(e2e_t)
    n_obs = rsum(float(st["n_obs"]))
    n_cand = rsum(float(st["n_candidates"]))
    pairs_eval = rsum(float(st["pairs_evaluated"]))
    stage_ms = {k: rmax(tot[k] / K) for k in tot}
    nodes = rsum(float(stc["nodes_visited"]))
    tris_t = rsum(float(stc["tris_tested"]))
    if ex is not None:
        ex_t = rmax(ex[0]["ms_total"] / 1e3 / ex[2])
        ex_cull = rmax(ex[0]["ms_cull"] / ex[2])

    trace("reductions done")
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- parity of the e2e result against the oracle's CPU arm (and the CPU baseline at N = 1) ----------------
    cpu_line = None
    parity = None
    if not args.no_cpu_baseline:
        if world == 1:
            v, cores, sample, _, sidx, svis = cpu_arm(prob.cams, prob.pts, prob.xyz, prob.tri, 12.0)
            cpu_line = {"value": v, "unit": "tests/s", "cores": cores, "kind": "port", "sample": sample,
                        "build": "-O3 -march=native -fopenmp, on this box"}
        else:
            _, _, _, _, sidx, svis = cpu_arm(prob.cams, prob.pts, prob.xyz, prob.tri, 0.0, fixed_n=8 * world)
        parity = parity_against(sidx, svis, *csr)
    exp = expected_hash(args.workload)
    hash_line = {"value": f"0x{res_hash:016x}", "expected": f"0x{exp:016x}" if exp is not None else None,
                 "ok": (res_hash == exp) if exp is not None else None, "observations": n_obs_e2e,
                 "note": "order-sensitive hash of the ONE host CSR the e2e call returned; additive over cameras, so "
                         "the same at every N; expected = tests/golden/result_hashes.json (the N = 1 result)"}

    peak, peak_kind = measured_peaks()
    value = C * P * K / t_dev_max
    e2e_value = C * P * K / e2e_max
    # algorithmic bytes per stage (DESIGN.md "roofline bookkeeping"), whole job, per step
    n_words = (n_cand + 31) // 32
    nodes_per_cam_sum = nodes / max(1.0, n_cand / 32.0) * C if n_cand else 0.0  # ~ one list per camera
    if args.cull_mode == "grid":
        # fused grid schedule (DESIGN.md section 4): plan -> one fused pass per camera -> sort + write
        b_cull = 144.0 * C + 4.0 * C * 2 + 4.0 * nodes_per_cam_sum  # plan: camera + centre, count + offset;
        #                                                            leaf lists written (4 B per entry)
        b_trav = (24.0 * pairs_eval + 4.0 * n_cand + 144.0 * C      # grid-ordered point per evaluated pair,
                  + 36.0 * nodes + 48.0 * tris_t + 4.0 * n_obs)     # index per candidate, camera; list entry (4)
        #            + leaf box (32) per entry examined, 48 B record per warp-triangle test, scratch index out
        b_sort = 0.0
        b_comp = 4.0 * n_obs + 24.0 * n_obs + 20.0 * n_obs + 128.0 * C
        #        scratch index read, point gather, CSR record written, camera record + offsets
    else:
        # exhaustive schedule: every pair -> pool (key, uv) -> radix sort -> ordered traversal -> compaction
        b_cull = 24.0 * pairs_eval / 64.0 + 144.0 * C + 28.0 * n_cand  # a 64-camera tile reads each point once
        b_trav = 56.0 * n_cand + 32.0 * nodes + 48.0 * tris_t + 4.0 * n_words
        b_sort = 24.0 * n_cand * max(1, -(-(int(np.ceil(np.log2(max(C // world, 2)))) + int(np.ceil(np.log2(P)))) // 8))
        b_comp = 12.0 * n_cand + 8.0 * n_words + 24.0 * n_obs * 2 + 8.0 * (C + 1)
    b_prep = 24.0 * P * 2 + 28.0 * P + 8.0 * P  # grid build: SoA points read twice (count, fill), grid copy written, cell ids
    stages = {
        "prep": (b_prep * world, stage_ms["ms_prep"]),
        "cull": (b_cull, stage_ms["ms_cull"]), "sort": (b_sort, stage_ms["ms_sort"]),
        "traverse": (b_trav, stage_ms["ms_traverse"]), "compact": (b_comp, stage_ms["ms_compact"]),
    }
    dom = max(stages, key=lambda k: stages[k][1])
    ach = stages[dom][0] / (stages[dom][1] * 1e-3) / 1e9 if stages[dom][1] > 0 else 0.0
    kernel_of = ({"prep": "k_grid_count + k_grid_fill", "cull": "k_cam_plan + k_cam_trilist",
                  "traverse": "k_visibility_fused (cull + ray build + occlusion)",
                  "compact": "k_sort_write", "sort": "-"} if args.cull_mode == "grid" else
                 {"prep": "-", "cull": "k_cull_exhaustive", "sort": "k_rs_scatter (radix sort)", "traverse": "k_traverse",
                  "compact": "k_compact_write"})
    traffic, traffic_src = ncu_traffic(dom, args.workload, args.cull_mode)
    line = {
        "metric": "camera-point visibility tests/sec", "value": value, "unit": "tests/s",
        "n_gpus": world, "steps": K, "warmup": args.warmup, "ms_per_step": 1e3 * t_dev_max / K,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {
            "workload": describe(args.workload, C, P),
            "cameras": C, "points": P, "triangles": int(len(prob.tri)), "bvh_nodes": prob.scene.num_nodes,
            "cull_mode": args.cull_mode, "parallelism": f"camera ranges over {world} GPU(s), mesh/BVH/points replicated"
                           + ("; e2e: one process (rank 0) drives all GPUs through c2b_visibility_graph_multi: "
                              "points uploaded 1/N per GPU + ncclAllGather, one ncclAllGather of counts, one host CSR" if world > 1 else ""),
            "l2": "256 MB buffer written between timed steps (L2 flush)",
            "grid": "point grid dropped before every timed step: its build is inside value",
            "candidates": int(n_cand), "observations": int(n_obs),
            "pairs_evaluated_per_step": int(pairs_eval),
        },
        "value_cached_grid": {"value": C * P * K / t_cached_max, "ms_per_step": 1e3 * t_cached_max / K,
                              "note": "point grid kept between calls (same points, same max_dist)"},
        "observations_per_s": n_obs * K / t_dev_max,
        "evaluated_pairs_per_s": pairs_eval * K / t_dev_max,
        "e2e": {"value": e2e_value, "unit": "tests/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * e2e_max / K,
                "observations_per_s": n_obs_e2e * K / e2e_max, "stage_ms_last_step": e2e_stage,
                "inputs": "pinned host arrays", "entry": "c2b_visibility_graph" if world == 1 else "c2b_visibility_graph_multi"},
        "gpu_launches": int(launches_per_step * K),
        "stage_ms": {k: round(v, 4) for k, v in stage_ms.items()},
        "roofline": {
            "bound": "hbm", "stage": dom, "kernel": kernel_of[dom], "achieved": ach, "peak": peak * world, "unit": "GB/s",
            "frac": ach / (peak * world), "traffic": traffic, "traffic_source": traffic_src, "peak_kind": f"of {peak_kind} (MEASURED_PEAKS.json hbm_gbs x n_gpus)",
            "algorithmic_bytes_per_step": stages[dom][0],
            "all_stages_GBps": {k: (v[0] / (v[1] * 1e-3) / 1e9 if v[1] > 0 else None) for k, v in stages.items()},
            "warp_node_visits": int(nodes), "warp_triangle_tests": int(tris_t),
            # the whole pass by BASELINE.md section 5's single formula (node visits and triangle tests are
            # per 32-ray packet here: one fetch serves the packet)
            "pipeline": (lambda b: {"algorithmic_bytes_per_step": b, "achieved": b / (t_dev_max / K) / 1e9,
                                    "frac": b / (t_dev_max / K) / 1e9 / (peak * world),
                                    "formula": "24*pairs_evaluated + 120*C + 64*node_visits + 48*triangle_tests + 24*O + 8*(C+1)"})(
                24.0 * pairs_eval + 120.0 * C + 64.0 * nodes + 48.0 * tris_t + 24.0 * n_obs + 8.0 * (C + 1)),
        },
        "clocks": clocks,
        "result_hash": hash_line,
    }
    if parity is not None:
        line["parity"] = parity
    if multi_stats is not None:
        line["e2e"]["per_gpu_last_step"] = multi_stats
    line.update(extras)
    if noise is not None:
        line["noise"] = noise
    if ex is not None:
        line["exhaustive"] = {"value": C * P / ex_t, "unit": "tests/s", "ms_per_step": 1e3 * ex_t,
                              "cull_ms": ex_cull, "steps": ex[2],
                              "note": "every camera x point pair tested on the GPU (the reference's loop)"}
        # secondary bound (SURVEY 8d): the exhaustive cull's hot loop issues 7 FP64-pipe instructions per
        # pair (3 DADD + DMUL + 2 DFMA + DSETP); the probe is a loop of independent DFMAs on the same device
        rate = Ct.c_double(0.0)
        if L.c2b_probe_fp64(ctx.handle, Ct.byref(rate)) == 0 and rate.value > 0 and ex_cull > 0:
            per_rank_pairs = C * P / world
            line["exhaustive"]["fp64_probe_dfma_per_s"] = rate.value
            line["exhaustive"]["fp64_pipe_frac"] = 7.0 * per_rank_pairs / (ex_cull * 1e-3) / rate.value
    if cpu_line is not None:
        line["cpu_baseline"] = cpu_line

    # ---- the other single-GPU configurations, briefly (default run at N = 1 only) ------------------------------
    if default_run and world == 1 and not args.no_secondary:
        sec = {}
        prob.scene.close()
        del prob
        for name in ("cfg3", "cfg5"):
            p2 = Problem(name)
            t2, s2 = p2.resident(args.cull_mode, 5, 2)
            te, o5 = p2.e2e_single(5, 2, p2.pin_cams.data_ptr(), p2.pin_pts.data_ptr())
            O5 = int(o5.n_obs)
            h5 = result_hash(np.ctypeslib.as_array(o5.offsets, shape=(p2.C + 1,)),
                             np.ctypeslib.as_array(o5.point_idx, shape=(max(O5, 1),))[:O5],
                             np.ctypeslib.as_array(o5.uv, shape=(max(2 * O5, 1),))[:2 * O5])
            e5 = expected_hash(name)
            sec[name] = {"workload": describe(name, p2.C, p2.P), "triangles": int(len(p2.tri)),
                         "scene_build_ms": p2.scene_build_ms,
                         "ms_per_step": t2["ms_total"] / 5, "value": p2.C * p2.P * 5 / (t2["ms_total"] / 1e3),
                         "stage_ms": {k: round(t2[k] / 5, 4) for k in STAGES},
                         "e2e_ms_per_step": 1e3 * te / 5, "e2e_value": p2.C * p2.P * 5 / te,
                         "observations": O5, "result_hash": f"0x{h5:016x}",
                         "result_hash_ok": (h5 == e5) if e5 is not None else None}
            p2.scene.close()
            del p2
        line["secondary"] = sec
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *csr)
    real_stdout.write(json.dumps(line) + "\n")
    real_stdout.flush()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
