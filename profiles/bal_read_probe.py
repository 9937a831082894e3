"""BAProblem::from_file on the GPU (c2b_read_bal_resident) against the host readers, on the synthetic cities cfg3
and cfg4 with mesh occlusion, built as bench.py builds them.

For each config: upload -> resident visibility pass -> resident cull -> the GPU writer's .bal and .bbal in a fresh
temporary directory on local disk.  Then for each file: one warm-up read and N timed c2b_read_bal_resident calls on
the same ctx, split into pread(2) (host time), chunk copies and parse kernels (device time, CUDA events) by
c2b_bal_read_stats, plus the host wall time of the call, slow_tokens and regrouped; the C++ mirror's
BAProblem::from_file (a small program compiled from include/city2ba.hpp, steady clock around the call) and, on
cfg3, the Python mirror's from_file; and whether the downloaded problem equals the C++ mirror's bit for bit.  The
file is in the page cache for every read after the writer's (read(2) measures a memory copy, not the disk).

Algorithmic bytes of one read: the file crosses PCIe and is read from HBM once, the problem is written once
(8 (C + 1) + 20 O + 24 P + 72 C), text adds the camera column (4 O written and read) and, when the file is not in
camera order, the regroup (8 O).

    python profiles/bal_read_probe.py [--repeats 3] [--configs cfg3,cfg4] [--out FILE.json]
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

CPP = r"""
#include <chrono>
#include <cstdio>
#include <fstream>
#include "city2ba.hpp"
using namespace city2ba;
int main(int argc, char **argv) {  // BAL path, raw dump path
  auto t0 = std::chrono::steady_clock::now();
  const BAProblem ba = BAProblem::from_file(argv[1]);
  auto t1 = std::chrono::steady_clock::now();
  std::ofstream f(argv[2], std::ios::binary);
  const uint64_t n[3] = {ba.cameras.size(), ba.points.size(), ba.num_observations()};
  f.write((const char *)n, sizeof n);
  for (const auto &c : ba.cameras) f.write((const char *)c.rec, sizeof c.rec);
  for (const auto &p : ba.points) f.write((const char *)p.data(), 24);
  uint64_t o = 0;
  f.write((const char *)&o, 8);
  for (const auto &v : ba.vis_graph) {
    o += v.size();
    f.write((const char *)&o, 8);
  }
  for (const auto &v : ba.vis_graph)
    for (const auto &e : v) {
      const uint32_t p = (uint32_t)e.first;
      f.write((const char *)&p, 4);
    }
  for (const auto &v : ba.vis_graph)
    for (const auto &e : v) f.write((const char *)&e.second, 16);
  std::printf("{\"from_file_s\": %.6f}\n", std::chrono::duration<double>(t1 - t0).count());
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


def build_cpp(tmp):
    src, exe = os.path.join(tmp, "bal_read_mirror.cpp"), os.path.join(tmp, "bal_read_mirror")
    open(src, "w").write(CPP)
    so_dir = os.path.join(ROOT, "city2ba_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
                           "-L", so_dir, "-lcity2ba_cuda", f"-Wl,-rpath,{so_dir}"])
    return exe


def load_dump(path):
    d = open(path, "rb").read()
    C, P, O = np.frombuffer(d, np.uint64, 3).tolist()
    at = 24
    cams = np.frombuffer(d, np.float64, 15 * C, at).reshape(-1, 15)
    at += 120 * C
    pts = np.frombuffer(d, np.float64, 3 * P, at).reshape(-1, 3)
    at += 24 * P
    off = np.frombuffer(d, np.uint64, C + 1, at)
    at += 8 * (C + 1)
    idx = np.frombuffer(d, np.uint32, O, at)
    at += 4 * O
    uv = np.frombuffer(d, np.float64, 2 * O, at)
    return cams, pts, off, idx, uv


def timed_reads(c2b, ctx, path, repeats):
    rp = c2b.generate.ResidentProblem(ctx)
    rp.read(path)  # warm-up: the first read allocates its buffers
    runs = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        st = rp.read(path)
        st["wall_ms"] = (time.perf_counter() - t0) * 1e3
        runs.append(st)
    med = lambda k: float(np.median([r[k] for r in runs]))  # noqa: E731
    out = {k: runs[0][k] for k in ("n_cameras", "n_points", "n_obs", "bytes", "chunks", "slow_tokens", "regrouped")}
    out.update({k: med(k) for k in ("ms_read", "ms_h2d", "ms_parse", "wall_ms")})
    out["wall_ms_min"] = float(np.min([r["wall_ms"] for r in runs]))
    out["repeats"] = repeats
    return rp, out


def bits(a):
    return np.ascontiguousarray(a, np.float64).reshape(-1).view(np.uint64)


def probe(name, repeats, ctx, c2b, bench, tmp, exe, python_reader):
    cams, pts, xyz, tri = bench.build_workload(name)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    rp = c2b.generate.ResidentProblem(ctx)
    rp.upload_cameras(cams)
    rp.upload_points(pts)
    rp.run(scene, bench.MAX_DIST)
    st = rp.cull()
    C, P, O = st["n_cameras"], st["n_points"], st["n_obs"]
    rec = {"config": bench.describe(name, len(cams), len(pts)) + ", mesh occlusion, after the resident cull",
           "n_cameras": C, "n_points": P, "n_obs": O, "files": {}}
    for fmt in ("bal", "bbal"):
        path = os.path.join(tmp, f"{name}.{fmt}")
        rp.write(path)
        r, g = timed_reads(c2b, ctx, path, repeats)
        problem = {"bytes": 8 * (C + 1) + 20 * O + 24 * P + 72 * C}
        alg = g["bytes"] + problem["bytes"] + (8 * O if fmt == "bal" else 0) + (8 * O if g["regrouped"] else 0)
        g["algorithmic_hbm_bytes"] = alg
        g["parse_hidden_behind_copy"] = g["ms_parse"] <= g["ms_h2d"]
        c, p = r.download_problem(C, P)
        gr = r.download()
        raw = os.path.join(tmp, "cpp.raw")
        cpp = json.loads(subprocess.run([exe, path, raw], capture_output=True, text=True, check=True).stdout)
        cc, cp_, coff, cidx, cuv = load_dump(raw)
        os.remove(raw)
        g["cpp_mirror"] = {**cpp, "what": "include/city2ba.hpp BAProblem::from_file (operator>> / ifstream::read), "
                                          "one thread"}
        g["identical_to_cpp"] = bool(np.array_equal(coff, gr.offsets) and np.array_equal(cidx, gr.point_idx)
                                     and np.array_equal(bits(cuv), bits(gr.uv)) and np.array_equal(bits(cp_), bits(p))
                                     and np.array_equal(bits(cc), bits(c)))
        if python_reader:
            t0 = time.perf_counter()
            py = c2b.BAProblem.from_file(path)
            g["python_mirror"] = {"from_file_s": time.perf_counter() - t0,
                                  "what": "city2ba_b200.BAProblem.from_file"}
            g["identical_to_python_without_cameras"] = bool(
                np.array_equal(py.vis_graph.offsets, gr.offsets) and np.array_equal(py.vis_graph.point_idx, gr.point_idx)
                and np.array_equal(bits(py.vis_graph.uv), bits(gr.uv)) and np.array_equal(bits(py.points), bits(p)))
            del py
        rec["files"][fmt] = g
        os.remove(path)
    scene.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--configs", default="cfg3,cfg4")
    ap.add_argument("--python-reader", default="cfg3", help="configs on which the Python mirror is timed too")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import bench
    import city2ba_b200 as c2b
    ctx = c2b.context(0)
    tmp = tempfile.mkdtemp(prefix="bal_read_probe_")
    try:
        exe = build_cpp(tmp)
        rec = {"probe": "bal_read_probe", "device": device_info(), "results": []}
        for name in a.configs.split(","):
            r = probe(name, a.repeats, ctx, c2b, bench, tmp, exe, name in a.python_reader.split(","))
            print(json.dumps({"config": r["config"], "identical_to_cpp": {k: v["identical_to_cpp"]
                                                                            for k, v in r["files"].items()}}), flush=True)
            rec["results"].append(r)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    txt = json.dumps(rec, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(txt)
    print(txt)
    if not all(f["identical_to_cpp"] and f.get("identical_to_python_without_cameras", True)
               for r in rec["results"] for f in r["files"].values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
