"""noise::join_landmarks on the GPU (c2b_join_landmarks_resident) against the C++ host mirror, on the synthetic city
cfg4 with mesh occlusion, built as bench.py builds it, then culled.

1. Resident visibility pass, resident cull.  For each join_percent in {1e-3, 1e-2, 1e-1}: one warm-up call and N timed
   calls (each on the same culled graph, re-installed from a .bbal between calls), device ms from the stats (CUDA
   events on the ctx stream around the whole pass) and host wall ms around the call.
2. The split of one call per join_percent into index build (bounds, Morton codes, sort, tree, refit, layout),
   selection (radix-select histograms and the list) and queries (the sort of the selections by Morton position and
   k_jn_query), from a torch.profiler run of its own: the CUDA kernels and memsets of the call in time order, cut at
   the last k_bvh_layout and at k_jn_list.
3. The C++ mirror's host join_landmarks (include/city2ba.hpp: k-d tree build + one walk per selection) on the same
   problem at the same sizes, steady clock around the call, in a small program compiled here.
4. Parity at cfg3: the resident pass against the sequential restatement (tests/join_ref.c), point indices and counts.

5. The points' ties: how many points share their position with another point, and the largest such group (a query
   among coincident points visits every one of them: at distance 0 only the index decides, so no box is pruned).

    python profiles/join_probe.py [--repeats 5] [--config cfg4] [--resident-only] [--out FILE.json]

--resident-only runs steps 1, 2 and 5 (the bucket-size sweep of run_r03f.sh runs it once per prebuilt library).
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

PERCENTS = (1e-3, 1e-2, 1e-1)
PARITY_PERCENT = 2e-3

CPP = r"""
#include <chrono>
#include <cstdio>
#include "city2ba.hpp"
using namespace city2ba;
int main(int argc, char **argv) {  // .bbal in
  const BAProblem ba = BAProblem::from_file(argv[1]);
  for (double p : {%PERCENTS%}) {
    auto t0 = std::chrono::steady_clock::now();
    const BAProblem out = noise::join_landmarks(ba, p, 7);
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    std::printf("{\"join_percent\": %g, \"ms\": %.3f, \"n_obs\": %zu}\n", p, ms, out.num_observations());
    std::fflush(stdout);
  }
  return 0;
}
"""


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"name": None, "power_limit": None, "error": str(e)}


def stage_split(rp, src, p, seed):
    """device ms of the index build, the selection and the queries of one call (torch.profiler, CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    rp.read(src)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rp.join_landmarks(p, seed)
    ev = sorted((e for e in prof.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start)
    names = [e.name for e in ev]
    i_layout = max(i for i, n in enumerate(names) if "k_bvh_layout" in n)
    i_list = max(i for i, n in enumerate(names) if "k_jn_list" in n)
    ms = lambda es: sum(e.time_range.end - e.time_range.start for e in es) / 1e3  # noqa: E731  (us -> ms)
    per_kernel = {}
    for e in ev:
        per_kernel[e.name.split("(")[0]] = per_kernel.get(e.name.split("(")[0], 0.0) + (e.time_range.end - e.time_range.start) / 1e3
    return {"index_ms": ms(ev[:i_layout + 1]), "select_ms": ms(ev[i_layout + 1:i_list + 1]),
            "query_ms": ms(ev[i_list + 1:]), "kernels": len(ev),
            "query_kernel_ms": ms(e for e in ev if "k_jn_query" in e.name),
            "per_kernel_ms": {k: round(v, 4) for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1])},
            "source": "torch.profiler CUDA kernel + memset durations of one call, summed per stage"}


def split_or_error(rp, src, p, seed):
    try:
        return stage_split(rp, src, p, seed)
    except Exception as e:  # noqa: BLE001  (the split is a diagnostic: the pass times above stand without it)
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--config", default="cfg4")
    ap.add_argument("--resident-only", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import bench
    import city2ba_b200 as c2b
    ctx = c2b.context(0)
    rec = {"probe": "join_probe", "device": device_info()}
    tmp = tempfile.mkdtemp(prefix="c2b_join_probe_")
    try:
        cams, pts, xyz, tri = bench.build_workload(a.config)
        scene = c2b.Scene(xyz, tri, ctx=ctx)
        rp = c2b.generate.ResidentProblem(ctx)
        rp.upload_cameras(cams)
        rp.upload_points(pts)
        rp.run(scene, bench.MAX_DIST)
        st = rp.cull()
        scene.close()
        src = os.path.join(tmp, "culled.bbal")
        rp.write(src)
        rec["config"] = bench.describe(a.config, len(cams), len(pts)) + ", mesh occlusion, culled"
        rec["problem"] = {"n_cameras": st["n_cameras"], "n_points": st["n_points"], "n_obs": st["n_obs"]}
        seed = 11
        rows = []
        for p in PERCENTS:
            rp.read(src)
            rp.join_landmarks(p, seed)  # warm-up: the first call grows its buffers
            dev, wall, s = [], [], None
            for _ in range(a.repeats):
                rp.read(src)
                t0 = time.perf_counter()
                s = rp.join_landmarks(p, seed)
                wall.append((time.perf_counter() - t0) * 1e3)
                dev.append(s["ms_compute"])
            rows.append({"join_percent": p, "n_selected": s["n_selected"], "n_changed": s["n_changed"],
                         "gpu_ms": {"median": float(np.median(dev)), "min": float(np.min(dev)),
                                    "max": float(np.max(dev)), "repeats": a.repeats,
                                    "source": "CUDA events on the ctx stream around the pass"},
                         "gpu_wall_ms": {"median": float(np.median(wall)), "source": "host clock around the call"},
                         "split": split_or_error(rp, src, p, seed)})
            print(json.dumps(rows[-1]), flush=True)
        rec["resident"] = rows
        _, cpts = rp.download_problem(st["n_cameras"], st["n_points"])
        _, cnt = np.unique(cpts, axis=0, return_counts=True)
        rec["ties"] = {"points_sharing_a_position": int(np.sum(cnt[cnt > 1])), "largest_group": int(cnt.max()),
                       "positions": int(len(cnt))}
        print(json.dumps(rec["ties"]), flush=True)
        if not a.resident_only:
            # the C++ mirror's host form
            cpp = CPP.replace("%PERCENTS%", ", ".join(map(repr, PERCENTS)))
            open(os.path.join(tmp, "j.cpp"), "w").write(cpp)
            exe, so_dir = os.path.join(tmp, "j"), os.path.join(ROOT, "city2ba_b200")
            subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), os.path.join(tmp, "j.cpp"),
                                   "-o", exe, "-L", so_dir, "-lcity2ba_cuda", f"-Wl,-rpath,{so_dir}"])
            out = subprocess.run([exe, src], capture_output=True, text=True, check=True)
            rec["host_mirror"] = [json.loads(x) for x in out.stdout.splitlines() if x.startswith("{")]
            for r, h in zip(rows, rec["host_mirror"]):
                r["host_over_resident"] = h["ms"] / r["gpu_ms"]["median"] if r["gpu_ms"]["median"] > 0 else None
            print(json.dumps(rec["host_mirror"]), flush=True)
            # parity with the restatement at cfg3
            from test_oracle_join import JoinRef
            ref = JoinRef(tmp)
            c3, p3, x3, t3 = bench.build_workload("cfg3")
            scene = c2b.Scene(x3, t3, ctx=ctx)
            r3 = c2b.generate.ResidentProblem(ctx)
            r3.upload_cameras(c3)
            r3.upload_points(p3)
            r3.run(scene, bench.MAX_DIST)
            s3 = r3.cull()
            scene.close()
            _, pts3 = r3.download_problem(s3["n_cameras"], s3["n_points"])
            g3 = r3.download()
            ref_idx, ref_st, err = ref.join_landmarks(pts3, g3.point_idx, PARITY_PERCENT, seed)
            got = r3.join_landmarks(PARITY_PERCENT, seed)
            gi = r3.download().point_idx
            rec["parity_cfg3"] = {"join_percent": PARITY_PERCENT, "n_points": s3["n_points"], "n_obs": s3["n_obs"],
                                  "n_selected": got["n_selected"], "n_changed": got["n_changed"],
                                  "ref_error": err, "stats_equal": (got["n_selected"], got["n_changed"]) ==
                                  (ref_st["n_selected"], ref_st["n_changed"]),
                                  "mismatches": int(np.sum(gi != ref_idx)) if len(gi) == len(ref_idx) else -1}
            print(json.dumps(rec["parity_cfg3"]), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    txt = json.dumps(rec, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(txt)
    print(txt)
    if a.resident_only:
        return
    p = rec["parity_cfg3"]
    if p["mismatches"] != 0 or not p["stats_equal"] or p["ref_error"] is not None:
        sys.exit(1)


if __name__ == "__main__":
    main()
