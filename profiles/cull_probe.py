"""BAProblem::cull on the GPU (c2b_cull_problem_resident) against the host mirror's BAProblem.cull(), on the
synthetic cities cfg3 and cfg4 with mesh occlusion, built as bench.py builds them.

For each config: upload -> resident visibility pass -> (warm-up cull) -> N timed repeats of [re-upload + resident
pass, then c2b_cull_problem_resident] -> download the un-culled graph once and time BAProblem.cull() on it ->
compare the GPU result with the host's (camera records, points, offsets, indices, (u, v) as raw bits).

Algorithmic bytes of one application of LCC + remove_singletons on (C, P, O) -> (C', P', O'):
    read the problem once        120 C + 24 P + 8 (C + 1) + 20 O
    write the result once        120 C' + 24 P' + 8 (C' + 1) + 20 O'
    point indices twice more     8 O          (union-find pass, flag pass)
    labels written and read      8 (C + P)
summed over the applications (their sizes from the host loop) and divided by the device time of the cull.

    python profiles/cull_probe.py [--repeats 12] [--configs cfg3,cfg4] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

HBM_GBS = 6547.5  # MEASURED_PEAKS.json hbm_gbs of the B200 pool (SURVEY.md section 2)


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"name": None, "power_limit": None, "error": str(e)}


def app_bytes(a, b):
    (C, P, O), (C2, P2, O2) = a, b
    return (120 * C + 24 * P + 8 * (C + 1) + 20 * O) + (120 * C2 + 24 * P2 + 8 * (C2 + 1) + 20 * O2) + 8 * O + 8 * (C + P)


def host_loop(ba):
    """BAProblem.cull() step by step: the sizes of every application"""
    sizes = [(ba.num_cameras(), ba.num_points(), ba.num_observations())]
    nc, npt = ba.num_cameras(), ba.num_points()
    culled = ba.largest_connected_component().remove_singletons()
    sizes.append((culled.num_cameras(), culled.num_points(), culled.num_observations()))
    while (culled.num_cameras(), culled.num_points()) != (nc, npt):
        nc, npt = culled.num_cameras(), culled.num_points()
        culled = culled.largest_connected_component().remove_singletons()
        sizes.append((culled.num_cameras(), culled.num_points(), culled.num_observations()))
    return culled, sizes


def bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


def probe(name, repeats, ctx, c2b, bench):
    cams, pts, xyz, tri = bench.build_workload(name)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    rp = c2b.generate.ResidentProblem(ctx)

    def fresh():
        rp.upload_cameras(cams)
        rp.upload_points(pts)
        rp.run(scene, bench.MAX_DIST)

    fresh()
    g = rp.download()
    before = (len(cams), len(pts), g.num_observations)
    rp.cull()  # warm-up: the first cull allocates its buffers
    ms_dev, ms_wall, st = [], [], None
    for _ in range(repeats):
        fresh()
        t0 = time.perf_counter()
        st = rp.cull()
        ms_wall.append((time.perf_counter() - t0) * 1e3)
        ms_dev.append(st["ms_compute"])
    gc, gp = rp.download_problem(st["n_cameras"], st["n_points"])
    gg = rp.download()

    ba = c2b.BAProblem(cams, pts, g)
    t0 = time.perf_counter()
    ref, sizes = host_loop(ba)  # BAProblem.cull(), recording the sizes of each application
    host_s = time.perf_counter() - t0
    identical = (bits(gc).tobytes() == bits(ref.cameras).tobytes() and bits(gp).tobytes() == bits(ref.points).tobytes()
                 and np.array_equal(gg.offsets, ref.vis_graph.offsets)
                 and np.array_equal(gg.point_idx.astype(np.uint64), ref.vis_graph.point_idx)
                 and bits(gg.uv).tobytes() == bits(ref.vis_graph.uv).tobytes()
                 and st["iterations"] == len(sizes) - 1)
    B = sum(app_bytes(sizes[i], sizes[i + 1]) for i in range(len(sizes) - 1))
    med = float(np.median(ms_dev))
    scene.close()
    return {
        "config": bench.describe(name, len(cams), len(pts)) + ", mesh occlusion",
        "before": {"n_cameras": before[0], "n_points": before[1], "n_obs": before[2]},
        "after": {"n_cameras": st["n_cameras"], "n_points": st["n_points"], "n_obs": st["n_obs"]},
        "iterations": st["iterations"],
        "applications_sizes": sizes,
        "gpu_ms": {"median": med, "min": float(np.min(ms_dev)), "max": float(np.max(ms_dev)),
                   "repeats": repeats, "source": "CUDA events on the ctx stream around the fixed-point loop"},
        "gpu_wall_ms": {"median": float(np.median(ms_wall)), "min": float(np.min(ms_wall)),
                        "max": float(np.max(ms_wall)), "source": "host clock around c2b_cull_problem_resident"},
        "host_s": host_s,
        "host_what": "city2ba_b200.BAProblem.cull() (numpy + scipy connected_components) on the downloaded graph",
        "identical": bool(identical),
        "algorithmic_bytes": B,
        "algorithmic_bytes_per_iteration": B / max(st["iterations"], 1),
        "achieved_gbs": B / (med * 1e-3) / 1e9 if med > 0 else None,
        "frac_of_hbm": (B / (med * 1e-3) / 1e9) / HBM_GBS if med > 0 else None,
        "hbm_gbs": HBM_GBS,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=12)
    ap.add_argument("--configs", default="cfg3,cfg4")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import bench
    import city2ba_b200 as c2b
    ctx = c2b.context(0)
    rec = {"probe": "cull_probe", "device": device_info(), "results": []}
    for name in a.configs.split(","):
        r = probe(name, a.repeats, ctx, c2b, bench)
        print(json.dumps({k: r[k] for k in ("config", "iterations", "gpu_ms", "host_s", "identical")}), flush=True)
        rec["results"].append(r)
    txt = json.dumps(rec, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(txt)
    print(txt)
    if not all(r["identical"] for r in rec["results"]):
        sys.exit(1)


if __name__ == "__main__":
    main()
