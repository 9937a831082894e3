"""CPU model of the plan's row trim (k_cam_plan / camera_row, c2b_fused.cuh) at cfg4: how many grid points the fused
pass reads, and in how many 32-point chunks, when the point grid's x cells are 1/k of the y / z side (c2b_tune
"grid_x_split").  Numpy only; no GPU and no CUDA library.

    python profiles/row_trim_model.py [--workload cfg4] [--sample 3000] [--splits 1 4 8 16]

The grid is built as build_grid (c2b_api.cu) builds it and each camera's rows are trimmed as camera_row trims them
(the ball, in front of the camera, the four image side planes); a sample of evenly spaced cameras is evaluated and
scaled to all cameras.  The f64 operations run in numpy's order, not through the device's explicit intrinsics, so an
edge cell can come out one off: the counts are a model (within ~1 % of the library's pairs_evaluated at k = 1), not
the library's numbers.  "passing" counts the evaluated pairs that pass the cull predicate (the same for every k).
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MAX_CELLS = 4194304.0  # 2^22


def centres(cams):
    R = cams[:, :9].reshape(-1, 3, 3).transpose(0, 2, 1)  # pc = R p + t, column-major records
    return -np.einsum("nji,nj->ni", R, cams[:, 9:12])     # -R^T t


def build_grid(pts, cen, max_dist, cell_factor, split):
    """the host logic of build_grid: lo, inverse cell sides (x, y / z), n, data bounds, the x side"""
    h = max_dist * cell_factor
    mn, mx = pts.min(0), pts.max(0)
    ext = mx - mn
    lo = mn.copy()

    def cells_at(hh, s):
        return np.prod([min(np.floor(ext[k] / (hh / s if k == 0 else hh)) + 1.0, 1e9) for k in range(3)])

    pad = max_dist + 1e-6 * (abs(max_dist) + np.abs(cen.min(0)) + np.abs(cen.max(0)))
    rlo, rhi = cen.min(0) - pad, cen.max(0) + pad
    a, b = np.fmax(mn, rlo), np.fmin(mx, rhi)
    frac = np.prod(np.where(ext > 0, np.where(a <= b, np.fmin((b - a) / np.where(ext > 0, ext, 1), 1), 0), 1))
    drop = cells_at(h, 1) > MAX_CELLS or frac < 0.7
    if drop:  # the cameras' reach only
        lo = np.where(a <= b, a, rlo)
        ext = np.where(a <= b, b - a, 0.0)
        mn, mx = lo.copy(), np.where(a <= b, b, lo)
    while split > 1 and cells_at(h, split) > MAX_CELLS:
        split //= 2
    while True:
        n = np.array([min(np.floor(ext[k] / (h / split if k == 0 else h)) + 1.0, 1e9) for k in range(3)]).astype(np.int64)
        if np.prod(n.astype(float)) <= MAX_CELLS:
            break
        h *= 1.5
    inv_h = 1.0 / h
    inv_hx = 1.0 / (h / split)
    return dict(lo=lo, inv=np.array([inv_hx, inv_h, inv_h]), n=n, min_c=mn, max_c=mx, hx=1.0 / inv_hx,
                drop=drop, rlo=rlo, rhi=rhi, split=split)


def coord(g, k, x):
    t = np.floor((np.asarray(x, float) - g["lo"][k]) * g["inv"][k])
    c = np.clip(np.nan_to_num(t, nan=0.0, posinf=1e18, neginf=-1e18), 0, g["n"][k] - 1)
    return c.astype(np.int64)


def bin_points(g, pts):
    keep = np.ones(len(pts), bool)
    if g["drop"]:
        keep = np.all((pts >= g["rlo"]) & (pts <= g["rhi"]), axis=1)
    p = pts[keep]
    cx, cy, cz = (coord(g, k, p[:, k]) for k in range(3))
    cell = (cz * g["n"][1] + cy) * g["n"][0] + cx
    order = np.argsort(cell, kind="stable")
    cs = np.zeros(int(np.prod(g["n"])) + 1, np.int64)
    np.cumsum(np.bincount(cell, minlength=len(cs) - 1), out=cs[1:])
    return cs, p[order]


def trim_halfspace(g, nx, ny, nz, off, xr, mag_floor, y0, y1, z0, z1, x0, x1, alive):
    my = 0.0 if ny == 0.0 else ny * (y0 if ny > 0.0 else y1)
    mz = 0.0 if nz == 0.0 else nz * (z0 if nz > 0.0 else z1)
    bmin = my + mz + off
    mag = np.abs(my) + np.abs(mz) + abs(off) + xr + mag_floor
    ok = np.isfinite(bmin)
    slack = 1e-9 * mag + 1e-300
    flat = ok & (xr <= slack)
    alive &= ~(flat & (bmin > 2.0 * slack))
    lin = ok & ~(xr <= slack)
    with np.errstate(all="ignore"):
        xlim = -(bmin - slack) / nx
    lin &= ~np.isnan(xlim)
    xs = 1e-9 * (np.abs(xlim) + g["hx"])
    with np.errstate(all="ignore"):
        xe = xlim + xs if nx > 0.0 else xlim - xs
    if nx > 0.0:
        alive &= ~(lin & (xe < g["lo"][0]))
        x1 = np.where(lin, np.minimum(x1, coord(g, 0, xe)), x1)
    else:
        alive &= ~(lin & (xe > g["max_c"][0]))
        x0 = np.where(lin, np.maximum(x0, coord(g, 0, xe)), x0)
    return x0, x1, alive & (x0 <= x1)


def camera_rows(g, cs, c, cc, max_dist):
    """(start, end) of every row of the camera, in the plan's order; None = no rows"""
    lo, hi = np.zeros(3, np.int64), np.zeros(3, np.int64)
    for k in range(3):
        eps = 1e-9 * (abs(cc[k]) + abs(max_dist)) + 1e-300
        a0, a1 = cc[k] - max_dist - eps, cc[k] + max_dist + eps
        if a0 > g["max_c"][k] or a1 < g["min_c"][k]:
            return None
        lo[k], hi[k] = coord(g, k, a0), coord(g, k, a1)
    h = 1.0 / g["inv"][1]
    Z, Y = np.meshgrid(np.arange(lo[2], hi[2] + 1), np.arange(lo[1], hi[1] + 1), indexing="ij")
    Y, Z = Y.ravel(), Z.ravel()
    sl = 1e-6 * h
    y0 = np.where(Y == 0, g["min_c"][1], g["lo"][1] + Y * h - sl)
    y1 = np.where(Y == g["n"][1] - 1, g["max_c"][1], g["lo"][1] + (Y + 1) * h + sl)
    z0 = np.where(Z == 0, g["min_c"][2], g["lo"][2] + Z * h - sl)
    z1 = np.where(Z == g["n"][2] - 1, g["max_c"][2], g["lo"][2] + (Z + 1) * h + sl)
    reach = abs(cc[0]) + abs(max_dist)
    x0, x1 = np.full(len(Y), lo[0]), np.full(len(Y), hi[0])
    dy = np.fmax(np.fmax(y0 - cc[1], cc[1] - y1), 0.0)
    dz = np.fmax(np.fmax(z0 - cc[2], cc[2] - z1), 0.0)
    rem = max_dist * max_dist * 1.000000001 - (dy * dy + dz * dz)
    alive = rem >= 0.0
    w = np.sqrt(np.fmax(rem, 0.0)) * 1.000000001 + 1e-9 * reach
    xa, xb = cc[0] - w, cc[0] + w
    alive &= ~((xa > g["max_c"][0]) | (xb < g["min_c"][0]))
    x0, x1 = np.maximum(x0, coord(g, 0, xa)), np.minimum(x1, coord(g, 0, xb))
    alive &= x0 <= x1
    f = c[12]
    planar = c[13] == 0.0 and c[14] == 0.0 and abs(f) < np.inf
    rmax = np.abs(c[:12]).max()
    span = abs(cc[0]) + abs(cc[1]) + abs(cc[2]) + 3.0 * abs(max_dist)
    mag_floor = ((abs(f) if planar else 0.0) + 1.0) * (rmax * (span + 1.0))
    x0, x1, alive = trim_halfspace(g, c[2], c[5], c[8], c[11], abs(c[2]) * reach, mag_floor, y0, y1, z0, z1, x0, x1,
                                   alive)
    if planar:
        for k in range(4):
            row, sf = k >> 1, (-f if k & 1 else f)
            nx, ny = sf * c[row] + c[2], sf * c[3 + row] + c[5]
            nz, off = sf * c[6 + row] + c[8], sf * c[9 + row] + c[11]
            x0, x1, alive = trim_halfspace(g, nx, ny, nz, off, abs(nx) * reach, mag_floor, y0, y1, z0, z1, x0, x1,
                                           alive)
    base = (Z * g["n"][1] + Y) * g["n"][0]
    x0c, x1c = np.clip(x0, 0, g["n"][0] - 1), np.clip(x1, 0, g["n"][0] - 1)
    start, end = cs[base + x0c], cs[base + x1c + 1]
    return np.where(alive, start, 0), np.where(alive, end, 0)


def passing(p, c, cc, max_dist):
    d = cc - p
    pc = p @ c[:9].reshape(3, 3) + c[9:12]  # row k of R is (c[k], c[3 + k], c[6 + k])
    ok = (np.einsum("ij,ij->i", d, d) < max_dist * max_dist) & (pc[:, 2] <= 0.0)
    with np.errstate(all="ignore"):
        q = -pc[:, :2] / pc[:, 2:3]
        m2 = (q * q).sum(1)
        uv = (c[12] * (1.0 + c[13] * m2 + c[14] * m2 * m2))[:, None] * q
    return int((ok & np.all(np.abs(uv) <= 1.0, axis=1)).sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg4")
    ap.add_argument("--sample", type=int, default=3000)
    ap.add_argument("--splits", type=int, nargs="+", default=[1, 4, 8, 16])
    args = ap.parse_args()
    import bench
    cams, pts, _, _ = bench.build_workload(args.workload, gen="oracle")
    cams, pts = np.asarray(cams, float), np.asarray(pts, float)
    cen = centres(cams)
    max_dist = bench.MAX_DIST
    sample = np.unique(np.linspace(0, len(cams) - 1, args.sample).astype(np.int64))
    scale = len(cams) / len(sample)
    print(f"{args.workload}: {len(cams)} cameras, {len(pts)} points, max_dist {max_dist}; "
          f"{len(sample)} cameras sampled, counts scaled by {scale:.2f}")
    print("| x split k | pairs evaluated | passing | 32-point chunks, one row per chunk | chunks packed across rows |")
    print("|---|---|---|---|---|")
    for k in args.splits:
        g = build_grid(pts, cen, max_dist, 0.25, k)
        cs, gp = bin_points(g, pts)
        pairs = one_row = packed = passed = 0
        for i in sample:
            rows = camera_rows(g, cs, cams[i], cen[i], max_dist)
            if rows is None:
                continue
            start, end = rows
            n = np.maximum(end - start, 0)
            pairs += int(n.sum())
            one_row += int(((n + 31) // 32).sum())
            for b in range(0, len(n), 32):  # the fused pass packs each block of 32 rows
                packed += int((n[b:b + 32].sum() + 31) // 32)
            if n.any():
                idx = np.concatenate([np.arange(s, e) for s, e in zip(start, end) if e > s])
                passed += passing(gp[idx], cams[i], cen[i], max_dist)
        label = f"{k}" if g["split"] == k else f"{k} (capped to {g['split']})"
        print(f"| {label} | {pairs * scale / 1e6:.1f} M | {passed * scale / 1e6:.1f} M | {one_row * scale / 1e6:.2f} M "
              f"| {packed * scale / 1e6:.2f} M |", flush=True)


if __name__ == "__main__":
    main()
