"""SASS of a kernel of libcity2ba_cuda.so, attributed to source lines (-lineinfo) and summed per source FUNCTION:
static instruction counts per section of the hot loop, the opcode mix, and the lines that prove the claims made in
DESIGN.md (REDUX packet reductions, LDS.128 record reads, MATCH-based ranks, no spills in the inner loops).

    python profiles/sass_sections.py [kernel-substring] > profiles/<tag>_sass_fused.txt
"""
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "city2ba_b200", "libcity2ba_cuda.so")
KERNEL = sys.argv[1] if len(sys.argv) > 1 else "k_visibility_fusedILi0ELb0ELi4ELb0E"   # <MESH, no count, 4 CTAs, no walk>


def functions_of(path):
    """[(first line, last line, name)] of the __device__ / __global__ / C2B_HD functions of a source file"""
    out, cur = [], None
    pat = re.compile(r"^(?:template\s*<[^>]*>\s*)?(?:__device__|__global__|C2B_HD|static|inline)[^;{]*?\b([A-Za-z_][A-Za-z0-9_]*)\s*\($")
    lines = open(path).read().split("\n")
    for i, ln in enumerate(lines, 1):
        m = re.search(r"\b(k_[A-Za-z0-9_]+)\s*\(", ln) if ln.startswith("__global__") else None
        m = m or re.match(r"^(?:__device__|__global__|C2B_HD)\b.*?\b([A-Za-z_][A-Za-z0-9_]*)\s*\(", ln) or \
            re.match(r"^__global__ void .*?\b([A-Za-z_][A-Za-z0-9_]*)\s*\(", ln) or \
            re.match(r"^\s*(?:__launch_bounds__\([^)]*\)\s*)?(k_[A-Za-z0-9_]*)\s*\(", ln)
        if m and not ln.startswith(" " * 4):
            if cur:
                out.append((cur[0], i - 1, cur[1]))
            cur = (i, m.group(1))
    if cur:
        out.append((cur[0], len(lines), cur[1]))
    return out


def main():
    tmp = tempfile.mkdtemp()
    subprocess.run(["cuobjdump", "-xelf", "all", SO], cwd=tmp, capture_output=True)
    cubin = [f for f in os.listdir(tmp) if f.startswith("c2b_api.") and f.endswith(".cubin")][0]
    sass = subprocess.run(["nvdisasm", "-g", "-c", os.path.join(tmp, cubin)], capture_output=True, text=True).stdout.split("\n")
    start = next(i for i, ln in enumerate(sass) if ln.startswith(".text.") and KERNEL in ln)
    end = next((i for i in range(start + 1, len(sass)) if sass[i].startswith("//--------------------- ")), len(sass))
    body = sass[start:end]
    fn_cache = {}
    per_fn = collections.Counter()
    per_fn_fp64 = collections.Counter()
    ops = collections.Counter()
    where = ("?", 0)
    n = 0
    proofs = collections.defaultdict(list)
    for ln in body:
        m = re.match(r'\s*//## File "([^"]+)", line (\d+)', ln)
        if m:
            where = (m.group(1), int(m.group(2)))
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P[0-9T]+\s+)?([A-Z][A-Z0-9_.]*)", ln)
        if not m:
            continue
        op = m.group(1)
        n += 1
        ops[op.split(".")[0]] += 1
        f, line = where
        if f not in fn_cache:
            fn_cache[f] = functions_of(f) if os.path.exists(f) else []
        name = next((nm for a, b, nm in fn_cache[f] if a <= line <= b), "?")
        key = f"{os.path.basename(f)}:{name}"
        per_fn[key] += 1
        if op.split(".")[0] in ("DADD", "DMUL", "DFMA", "DSETP", "DMNMX", "MUFU", "F2F", "I2F", "F2I"):
            per_fn_fp64[key] += 1
        for tag, pat in (("CREDUX (warp min / max reductions of the packet bounds)", r"^C?REDUX"), ("LDS.128", r"^LDS\.128"), ("MATCH", r"^MATCH"), ("local memory (spill)", r"^(LDL|STL)"),
                         ("ATOMG / RED", r"^(ATOMG|RED)\b"), ("LDG.E.128 (node / triangle fetch)", r"^LDG\.E\.128")):
            if re.match(pat, op):
                proofs[tag].append(f"{key} line {line}")
    print(f"kernel {KERNEL}: {n} SASS instructions ({16 * n / 1024:.0f} KB)")
    print("\nper source function (static instruction count; FP64-pipe / conversion instructions in brackets):")
    for k, v in per_fn.most_common():
        print(f"  {v:6d}  [{per_fn_fp64[k]:5d}]  {k}")
    print("\nopcode mix (top 24):")
    for k, v in ops.most_common(24):
        print(f"  {v:6d}  {k}")
    print("\nevidence:")
    for tag, lst in proofs.items():
        c = collections.Counter(x.split(" line ")[0] for x in lst)
        print(f"  {tag}: {len(lst)}  " + ", ".join(f"{k} x{v}" for k, v in c.most_common(6)))


if __name__ == "__main__":
    main()
