"""BAProblem::write on the GPU (c2b_write_bal_resident) against the host writers, on the synthetic cities cfg3 and
cfg4 with mesh occlusion, built as bench.py builds them.

For each config: upload -> resident visibility pass -> resident cull -> for text and binary: one warm-up write, then
N timed resident writes into a file on local disk (a fresh temporary directory) and N into /dev/null, each split
into encode / D2H (device time, CUDA events) and write(2) (host time) by c2b_bal_stats, plus the host wall time of
the call.  Then the same problem through the C++ mirror's write_text / write_binary (a small program compiled from
include/city2ba.hpp, timed with a steady clock around each call) and, on cfg3, the Python mirror's write_text /
write_binary.  Outputs are compared byte for byte: GPU vs C++ whole files (text only when every value is below 2^53
in magnitude, where std::to_chars(fixed) also prints the shortest digits), GPU vs Python outside the camera lines /
block (Python's to_vec may differ in the last bit).

Algorithmic HBM bytes of one encode: the file written once, plus the CSR read once (8 (C + 1) + 20 O), the points
(24 P) and the camera vectors (72 C).  Text also reads every observation's CSR slot twice (length pass and write
pass), which is counted.  Share of peak = those bytes / ms_encode against HBM_GBS.

    python profiles/bal_probe.py [--repeats 3] [--configs cfg3,cfg4] [--out FILE.json]
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

HBM_GBS = 6547.5  # MEASURED_PEAKS.json hbm_gbs of the B200 pool (SURVEY.md section 2)

CPP = r"""
#include <chrono>
#include <cstdio>
#include <fstream>
#include "city2ba.hpp"
using namespace city2ba;
int main(int argc, char **argv) {  // raw problem dump, text path, binary path
  std::ifstream f(argv[1], std::ios::binary);
  uint64_t n[3];
  f.read((char *)n, sizeof n);
  const uint64_t C = n[0], P = n[1], O = n[2];
  BAProblem ba;
  ba.cameras.resize(C);
  for (auto &c : ba.cameras) f.read((char *)c.rec, sizeof c.rec);
  ba.points.resize(P);
  for (auto &p : ba.points) f.read((char *)p.data(), 24);
  std::vector<uint64_t> off(C + 1);
  std::vector<uint32_t> idx(O);
  std::vector<double> uv(2 * O);
  f.read((char *)off.data(), 8 * (C + 1));
  f.read((char *)idx.data(), 4 * O);
  f.read((char *)uv.data(), 16 * O);
  ba.vis_graph.resize(C);
  for (uint64_t c = 0; c < C; ++c)
    for (uint64_t k = off[c]; k < off[c + 1]; ++k) ba.vis_graph[c].push_back({idx[k], {uv[2 * k], uv[2 * k + 1]}});
  auto t0 = std::chrono::steady_clock::now();
  ba.write_text(argv[2]);
  auto t1 = std::chrono::steady_clock::now();
  ba.write_binary(argv[3]);
  auto t2 = std::chrono::steady_clock::now();
  std::printf("{\"write_text_s\": %.6f, \"write_binary_s\": %.6f}\n", std::chrono::duration<double>(t1 - t0).count(),
              std::chrono::duration<double>(t2 - t1).count());
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
    src, exe = os.path.join(tmp, "bal_mirror.cpp"), os.path.join(tmp, "bal_mirror")
    open(src, "w").write(CPP)
    so_dir = os.path.join(ROOT, "city2ba_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
                           "-L", so_dir, "-lcity2ba_cuda", f"-Wl,-rpath,{so_dir}"])
    return exe


def dump(path, cams, pts, g):
    with open(path, "wb") as f:
        f.write(np.array([len(cams), len(pts), g.num_observations], np.uint64).tobytes())
        f.write(np.ascontiguousarray(cams, np.float64).tobytes())
        f.write(np.ascontiguousarray(pts, np.float64).tobytes())
        f.write(np.ascontiguousarray(g.offsets, np.uint64).tobytes())
        f.write(np.ascontiguousarray(g.point_idx, np.uint32).tobytes())
        f.write(np.ascontiguousarray(g.uv, np.float64).tobytes())


def resident_write(c2b, ctx, path, fmt):
    """c2b_write_bal_resident with an explicit format (/dev/null has no extension to dispatch on)"""
    import ctypes
    st = c2b._lib.BalStats()
    c2b._lib.check(c2b._lib.lib().c2b_write_bal_resident(ctx.handle, path.encode(), fmt, ctypes.byref(st)))
    return st.to_dict()


def timed_writes(c2b, ctx, path, fmt, repeats):
    resident_write(c2b, ctx, path, fmt)  # warm-up: the first write allocates its buffers
    runs = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        st = resident_write(c2b, ctx, path, fmt)
        st["wall_ms"] = (time.perf_counter() - t0) * 1e3
        runs.append(st)
    med = lambda k: float(np.median([r[k] for r in runs]))  # noqa: E731
    return {"bytes": runs[0]["bytes"], "chunks": runs[0]["chunks"], "ms_encode": med("ms_encode"),
            "ms_d2h": med("ms_d2h"), "ms_write": med("ms_write"), "wall_ms": med("wall_ms"),
            "wall_ms_min": float(np.min([r["wall_ms"] for r in runs])), "repeats": repeats}


def split_lines(data, C, O):
    lines = data.split(b"\n")
    return lines[:1 + O] + lines[1 + O + C:]


def probe(name, repeats, ctx, c2b, bench, tmp, exe, python_writer):
    cams, pts, xyz, tri = bench.build_workload(name)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    rp = c2b.generate.ResidentProblem(ctx)
    rp.upload_cameras(cams)
    rp.upload_points(pts)
    rp.run(scene, bench.MAX_DIST)
    st = rp.cull()
    C, P, O = st["n_cameras"], st["n_points"], st["n_obs"]
    rec = {"config": bench.describe(name, len(cams), len(pts)) + ", mesh occlusion, after the resident cull",
           "n_cameras": C, "n_points": P, "n_obs": O, "gpu": {}}
    files = {}
    for fmt in ("bal", "bbal"):
        disk = os.path.join(tmp, f"gpu.{fmt}")
        f = c2b._lib.BAL_TEXT if fmt == "bal" else c2b._lib.BAL_BINARY
        rec["gpu"][fmt] = {"disk": timed_writes(c2b, ctx, disk, f, repeats),
                           "dev_null": timed_writes(c2b, ctx, "/dev/null", f, repeats)}
        files[fmt] = open(disk, "rb").read()
        g = rec["gpu"][fmt]["disk"]
        hbm = g["bytes"] + 8 * (C + 1) + 20 * O + 24 * P + 72 * C + (8 * O if fmt == "bal" else 0)
        rec["gpu"][fmt]["algorithmic_hbm_bytes"] = hbm
        rec["gpu"][fmt]["encode_gbs"] = hbm / (g["ms_encode"] * 1e-3) / 1e9
        rec["gpu"][fmt]["encode_frac_of_hbm"] = rec["gpu"][fmt]["encode_gbs"] / HBM_GBS
    c, p = rp.download_problem(C, P)
    gr = rp.download()
    ba = c2b.BAProblem(c, p, gr)
    raw = os.path.join(tmp, "problem.raw")
    dump(raw, c, p, gr)
    ct, cb = os.path.join(tmp, "cpp.bal"), os.path.join(tmp, "cpp.bbal")
    r = json.loads(subprocess.run([exe, raw, ct, cb], capture_output=True, text=True, check=True).stdout)
    maxabs = float(max(np.abs(c).max(initial=0), np.abs(p).max(initial=0), np.abs(gr.uv).max(initial=0)))
    rec["cpp_mirror"] = {**r, "what": "include/city2ba.hpp BAProblem::write_text / write_binary (std::to_chars + "
                                     "ofstream), one thread"}
    rec["identical"] = {"binary_vs_cpp": open(cb, "rb").read() == files["bbal"],
                        "text_vs_cpp": open(ct, "rb").read() == files["bal"],
                        "text_vs_cpp_expected": maxabs < 2.0 ** 53}
    if python_writer:
        pt, pb = os.path.join(tmp, "py.bal"), os.path.join(tmp, "py.bbal")
        t0 = time.perf_counter()
        ba.write_text(pt)
        t1 = time.perf_counter()
        ba.write_binary(pb)
        t2 = time.perf_counter()
        rec["python_mirror"] = {"write_text_s": t1 - t0, "write_binary_s": t2 - t1,
                                "what": "city2ba_b200.BAProblem.write_text / write_binary"}
        s, e = 24 + 8 * C + 24 * O, 24 + 8 * C + 24 * O + 72 * C
        pyb = open(pb, "rb").read()
        rec["identical"]["text_vs_python_without_camera_lines"] = \
            split_lines(open(pt, "rb").read(), C, O) == split_lines(files["bal"], C, O)
        rec["identical"]["binary_vs_python_without_camera_block"] = pyb[:s] == files["bbal"][:s] and pyb[e:] == files["bbal"][e:]
        rec["identical"]["binary_camera_block_vs_python_bit_equal"] = pyb[s:e] == files["bbal"][s:e]
    scene.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--configs", default="cfg3,cfg4")
    ap.add_argument("--python-writer", default="cfg3", help="configs on which the Python mirror is timed too")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import bench
    import city2ba_b200 as c2b
    ctx = c2b.context(0)
    tmp = tempfile.mkdtemp(prefix="bal_probe_")
    try:
        exe = build_cpp(tmp)
        rec = {"probe": "bal_probe", "device": device_info(), "results": []}
        for name in a.configs.split(","):
            r = probe(name, a.repeats, ctx, c2b, bench, tmp, exe, name in a.python_writer.split(","))
            print(json.dumps({"config": r["config"], "identical": r["identical"]}), flush=True)
            rec["results"].append(r)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    txt = json.dumps(rec, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(txt)
    print(txt)
    ok = all(r["identical"]["binary_vs_cpp"] and (r["identical"]["text_vs_cpp"] or not r["identical"]["text_vs_cpp_expected"])
             and r["identical"].get("text_vs_python_without_camera_lines", True)
             and r["identical"].get("binary_vs_python_without_camera_block", True) for r in rec["results"])
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
