"""noise::add_incorrect_correspondences on the GPU (c2b_add_incorrect_correspondences_resident) against the C++ host
mirror, on the synthetic city cfg4 with mesh occlusion, built as bench.py builds it, then culled.

1. Resident visibility pass, resident cull.  For each mismatch_chance in {1e-5, 1e-2, 1e-1}: one warm-up call and N
   timed calls (each on the same culled graph, re-installed from a .bbal between calls), device ms from the stats
   (CUDA events around the pass) and host wall ms around the call.  Work: sum over the selected observations of their
   camera's length n_c, each selection walks its camera twice or three times (maximum, weight sum, prefix search).
   The selections are recomputed here from the Philox stream (numpy) and checked against n_selected.
2. The C++ mirror's host add_incorrect_correspondences (include/city2ba.hpp) on the same graph at 1e-5 and 1e-2,
   steady clock around the call, in a small program compiled here.
3. The default chain read .bbal -> drift -> noise -> mismatch (1e-2) -> write .bbal: resident (host clock around the
   calls, each ends in a device synchronisation) against its host form (the C++ mirror: from_file, add_drift_normalized
   and add_noise on host arrays through the library, the host mismatch, write).

    python profiles/mismatch_probe.py [--repeats 5] [--config cfg4] [--out FILE.json]
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
sys.dont_write_bytecode = True

CHANCES = (1e-5, 1e-2, 1e-1)
DRIFT = (0.01, 0.001, 0.1)
NOISE = (0.01, 0.001, 0.01, 0.001)
CHAIN_CHANCE = 1e-2

CPP = r"""
#include <chrono>
#include <cstdio>
#include "city2ba.hpp"
using namespace city2ba;
static double ms_since(std::chrono::steady_clock::time_point t0) {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}
int main(int argc, char **argv) {  // .bbal in, .bbal out
  const Context ctx(0);
  {
    const BAProblem ba = BAProblem::from_file(argv[1]);
    for (double p : {1e-5, 1e-2}) {
      auto t0 = std::chrono::steady_clock::now();
      const BAProblem out = noise::add_incorrect_correspondences(ba, p, 7);
      std::printf("{\"mirror\": %g, \"ms\": %.3f, \"n_obs\": %zu}\n", p, ms_since(t0), out.num_observations());
    }
  }
  auto t0 = std::chrono::steady_clock::now();
  BAProblem ba = BAProblem::from_file(argv[1]);
  const double t_read = ms_since(t0);
  auto t1 = std::chrono::steady_clock::now();
  ba = noise::add_drift_normalized(ctx, ba, %DRIFT%, 3);
  ba = noise::add_noise(ctx, ba, %NOISE%, 4);
  const double t_noise = ms_since(t1);
  auto t2 = std::chrono::steady_clock::now();
  ba = noise::add_incorrect_correspondences(ba, %CHANCE%, 5);
  const double t_mm = ms_since(t2);
  auto t3 = std::chrono::steady_clock::now();
  ba.write(argv[2]);
  const double t_write = ms_since(t3);
  std::printf("{\"chain_ms\": %.3f, \"read\": %.3f, \"drift_noise\": %.3f, \"mismatch\": %.3f, \"write\": %.3f}\n",
              ms_since(t0), t_read, t_noise, t_mm, t_write);
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


def selection_u(O, seed, chunk=1 << 23):
    """u = ((w0 | w1 << 32) >> 11) 2^-53 of every observation's Philox4x32-10 block (key seed, counter (o, 6, 0))"""
    M0, M1, mask = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0xffffffff)
    out = np.empty(O)
    for s in range(0, O, chunk):
        o = np.arange(s, min(O, s + chunk), dtype=np.uint64)
        c0, c1 = o & mask, o >> np.uint64(32)
        c2, c3 = np.full_like(o, 6), np.zeros_like(o)
        k0, k1 = seed & 0xffffffff, seed >> 32
        for _ in range(10):
            p0, p1 = M0 * c0, M1 * c2
            c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & mask, \
                (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & mask
            k0, k1 = (k0 + 0x9E3779B9) & 0xffffffff, (k1 + 0xBB67AE85) & 0xffffffff
        out[s:s + len(o)] = ((c1 << np.uint64(32) | c0) >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--config", default="cfg4")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import bench
    import city2ba_b200 as c2b
    ctx = c2b.context(0)
    rec = {"probe": "mismatch_probe", "device": device_info()}
    tmp = tempfile.mkdtemp(prefix="c2b_mismatch_probe_")
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
        g = rp.download()
        n = np.diff(g.offsets.astype(np.int64))
        cam_of = np.repeat(np.arange(len(n)), n)
        multi = n > 1
        rec["config"] = bench.describe(a.config, len(cams), len(pts)) + ", mesh occlusion, culled"
        rec["graph"] = {"n_cameras": st["n_cameras"], "n_points": st["n_points"], "n_obs": st["n_obs"],
                        "sum_nc2": int(np.sum(n[multi].astype(np.float64) ** 2)),
                        "mean_nc": float(n.mean()) if len(n) else 0.0, "max_nc": int(n.max()) if len(n) else 0}
        seed = 11
        u = selection_u(int(st["n_obs"]), seed)
        rows = []
        for p in CHANCES:
            sel = (u <= p) & multi[cam_of]
            evals = int(n[cam_of[sel]].astype(np.int64).sum())
            rp.read(src)
            rp.add_incorrect_correspondences(p, seed)  # warm-up: the first call grows its buffers
            dev, wall, s = [], [], None
            for _ in range(a.repeats):
                rp.read(src)
                t0 = time.perf_counter()
                s = rp.add_incorrect_correspondences(p, seed)
                wall.append((time.perf_counter() - t0) * 1e3)
                dev.append(s["ms_compute"])
            med = float(np.median(dev))
            rows.append({"mismatch_chance": p, "n_selected": s["n_selected"], "n_swapped": s["n_swapped"],
                         "selected_matches_philox": int(sel.sum()) == s["n_selected"],
                         "sum_selected_nc": evals,
                         "gpu_ms": {"median": med, "min": float(np.min(dev)), "max": float(np.max(dev)),
                                    "repeats": a.repeats, "source": "CUDA events on the ctx stream around the pass"},
                         "gpu_wall_ms": {"median": float(np.median(wall)), "source": "host clock around the call"},
                         "distance_evals_per_s": evals / (med * 1e-3) if med > 0 else None})
            print(json.dumps(rows[-1]), flush=True)
        rec["resident"] = rows
        # the C++ mirror, and the host form of the chain
        cpp = CPP.replace("%DRIFT%", ", ".join(map(repr, DRIFT))).replace("%NOISE%", ", ".join(map(repr, NOISE)))
        cpp = cpp.replace("%CHANCE%", repr(CHAIN_CHANCE))
        open(os.path.join(tmp, "m.cpp"), "w").write(cpp)
        exe, so_dir = os.path.join(tmp, "m"), os.path.join(ROOT, "city2ba_b200")
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), os.path.join(tmp, "m.cpp"),
                               "-o", exe, "-L", so_dir, "-lcity2ba_cuda", f"-Wl,-rpath,{so_dir}"])
        out = subprocess.run([exe, src, os.path.join(tmp, "host_chain.bbal")], capture_output=True, text=True, check=True)
        lines = [json.loads(x) for x in out.stdout.splitlines() if x.startswith("{")]
        rec["host_mirror"] = [x for x in lines if "mirror" in x]
        rec["host_chain"] = [x for x in lines if "chain_ms" in x][0]
        # the resident chain
        t = {}
        t0 = time.perf_counter()
        rp.read(src)
        t["read"] = (time.perf_counter() - t0) * 1e3
        t1 = time.perf_counter()
        rp.add_drift(*DRIFT, seed=3)
        rp.add_noise(*NOISE, seed=4)
        rp.reprojection_error(2.0)  # ends in a device synchronisation
        t["drift_noise"] = (time.perf_counter() - t1) * 1e3
        t2 = time.perf_counter()
        rp.add_incorrect_correspondences(CHAIN_CHANCE, seed=5)
        t["mismatch"] = (time.perf_counter() - t2) * 1e3
        t3 = time.perf_counter()
        rp.write(os.path.join(tmp, "resident_chain.bbal"))
        t["write"] = (time.perf_counter() - t3) * 1e3
        t["chain_ms"] = (time.perf_counter() - t0) * 1e3
        rec["resident_chain"] = t
        rec["chain_what"] = ("read .bbal -> add_drift_normalized%s -> add_noise%s -> add_incorrect_correspondences(%g) -> "
                             "write .bbal; the two forms draw differently (host mismatch: the mirror's Rng)"
                             % (DRIFT, NOISE, CHAIN_CHANCE))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    txt = json.dumps(rec, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(txt)
    print(txt)
    if not all(r["selected_matches_philox"] for r in rec["resident"]):
        sys.exit(1)


if __name__ == "__main__":
    main()
