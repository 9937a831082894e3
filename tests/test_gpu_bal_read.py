"""BAL files read on the GPU (c2b_read_bal_resident) against Python's float() and the host readers of both mirrors.

Every number the device reads must be the double Python's float() gives for the same token, bit for bit (NaN: the
quiet NaN with the token's sign), whatever its spelling or digit count.  Whole files must give the problem the Python
mirror's from_file_text / from_file_binary gives: the same CSR, (u, v) and points bit for bit, and camera records that
are c2b_camera_from_vec of the file's 9-vectors."""
import ctypes
import math
import os
import random
import struct
import subprocess
from decimal import Decimal, getcontext

import numpy as np
import pytest

from city2ba_b200.baproblem import IOError_, ParseError
from conftest import bits_equal
from test_gpu_bal import camera_vecs, random_problem, special_values

pytestmark = pytest.mark.gpu

INVALID = -1


def fbits(x):
    return struct.unpack("<Q", struct.pack("<d", x))[0]


def expected_bits(tok):
    """Python's float() of a token, with NaN as 0x7ff8000000000000 and the token's sign"""
    x = float(tok)
    if math.isnan(x):
        return 0xFFF8000000000000 if tok.startswith("-") else 0x7FF8000000000000
    return fbits(x)


def resident(c2b, ctx):
    return c2b.generate.ResidentProblem(ctx)


def read_points_file(c2b, ctx, path, tokens):
    """a file of P points whose coordinates are `tokens` (padded with "0"); returns (bits of the read values, stats)"""
    tokens = list(tokens) + ["0"] * ((-len(tokens)) % 3)
    P = len(tokens) // 3
    with open(path, "w") as f:
        f.write(f"0 {P} 0\n")
        for i in range(P):
            f.write(" ".join(tokens[3 * i:3 * i + 3]) + "\n")
    rp = resident(c2b, ctx)
    st = rp.read(path)
    assert (st["n_cameras"], st["n_points"], st["n_obs"]) == (0, P, 0)
    _, pts = rp.download_problem(0, P)
    return pts.reshape(-1).view(np.uint64)[:len(tokens)], tokens, st


def check_tokens(c2b, ctx, path, tokens):
    got, tokens, st = read_points_file(c2b, ctx, path, tokens)
    exp = np.array([expected_bits(t) for t in tokens], np.uint64)
    bad = np.nonzero(got != exp)[0]
    if len(bad):
        pytest.fail(f"{len(bad)} of {len(tokens)} tokens read differently from float(), e.g. "
                    f"{[(tokens[i][:60], hex(int(got[i])), hex(int(exp[i]))) for i in bad[:3]]}")
    return st


def writer_spelling(c2b, ctx, vals, path):
    """the GPU writer's tokens for `vals` (a points-only file), in order"""
    from test_gpu_bal import points_only
    ba, vals = points_only(c2b, vals)
    ba.write_gpu(path, ctx)
    return open(path).read().split()[3:], vals


# ---- numbers ---------------------------------------------------------------------------------------------------------
def test_numbers_writer_spelling(c2b, ctx, tmp_path):
    """special_values() and 10^6 random bit patterns as the writer spells them read back bit for bit"""
    rng = np.random.default_rng(21)
    v = np.concatenate([special_values(), rng.integers(0, 2 ** 64, 10 ** 6, dtype=np.uint64).view(np.float64)])
    toks, vals = writer_spelling(c2b, ctx, v, str(tmp_path / "w.bal"))
    st = check_tokens(c2b, ctx, str(tmp_path / "r.bal"), toks)
    print(f"writer spelling: {len(toks)} tokens, slow_tokens = {st['slow_tokens']}")


def test_numbers_python_spellings(c2b, ctx, tmp_path):
    rng = random.Random(22)
    toks = []
    for _ in range(60000):
        x = struct.unpack("<d", struct.pack("<Q", rng.getrandbits(64)))[0]
        if math.isnan(x) or math.isinf(x):
            continue
        toks += [repr(x), "%.17g" % x, "%.25e" % x, "%.40f" % x if abs(x) < 1e60 else "%.3e" % x]
    for e in range(-330, 311):
        toks += [f"1e{e}", f"9.999999999999999999999e{e}", f"-5E{e}", f"+.5e{e}"]
    toks += ["+1", "+0.5", ".5", "5.", "-.5", "5.e3", "E".join(["1", "+05"]), "1E+05", "1e-05", "0001.5", "000",
             "-0", "+0.0", "00.000e0", "0e999999999999999999", "1e-999999999999999999", "1e400", "-1e-400",
             "inf", "-Infinity", "+INF", "iNfInItY", "nan", "-NaN", "+nAn", "1.7976931348623157e308",
             "1.7976931348623158e308", "2.2250738585072011e-308", "4.9406564584124654e-324"]
    check_tokens(c2b, ctx, str(tmp_path / "p.bal"), toks)


def test_numbers_long_mantissas(c2b, ctx, tmp_path):
    """20 to 800 digits, exact halfway cases and their neighbours: correctly rounded, some through the host"""
    getcontext().prec = 3000
    rng = random.Random(23)
    toks = ["9007199254740993", "9007199254740993.000000000000000000001", "9007199254740992.99999999999999999999",
            "9007199254740995", "1.00000000000000011102230246251565404236316680908203125",
            "1.000000000000000111022302462515654042363166809082031250000000001"]
    half = format(Decimal(2) ** -1075, "f")  # 752 significant digits, exactly half the smallest subnormal
    toks += [half, half + "1", half[:-1] + "4" + "9" * 40, "-" + half + "000001"]
    top = format(Decimal(2) ** 1024 - Decimal(2) ** 970, "f")  # halfway between the largest double and 2^1024
    toks += [top, top + ".000000000000000000000000001", str(int(top) - 1)]
    for _ in range(3000):
        nd = rng.randint(20, 800)
        d = str(rng.randint(1, 9)) + "".join(rng.choice("0123456789") for _ in range(nd - 1))
        e = rng.randint(-340, 300)
        k = rng.randint(0, nd)
        toks.append((d[:k] or "0") + "." + d[k:] + f"e{e - (nd - k) + 17}")
    for _ in range(2000):  # halfway points of random doubles, with up to 767 digits
        x = struct.unpack("<d", struct.pack("<Q", rng.getrandbits(63)))[0]
        if math.isnan(x) or math.isinf(x) or x == 0:
            continue
        m = (Decimal(x) + Decimal(float(np.nextafter(x, math.inf)))) / 2
        toks.append(format(m, "e") if rng.random() < 0.5 else format(m, "f"))
    st = check_tokens(c2b, ctx, str(tmp_path / "long.bal"), toks)
    assert st["slow_tokens"] > 0


# ---- round trip and whole files --------------------------------------------------------------------------------------
def download(c2b, rp, st):
    cams, pts = rp.download_problem(st["n_cameras"], st["n_points"])
    return cams, pts, rp.download()


def test_round_trip(c2b, ctx, tmp_path):
    """GPU writer then GPU reader: the same points and (u, v) bit for bit, both formats"""
    rng = np.random.default_rng(24)
    sv = special_values()
    ba = random_problem(c2b, rng, 30, len(sv) // 3 + 1, 40)
    pts = np.concatenate([sv, rng.integers(0, 2 ** 64, 3 * len(ba.points) - len(sv), dtype=np.uint64).view(np.float64)])
    ba.points = pts.reshape(-1, 3)
    uv = ba.vis_graph.uv.reshape(-1)
    uv[:] = rng.integers(0, 2 ** 64, len(uv), dtype=np.uint64).view(np.float64)
    uv[:min(len(uv), len(sv))] = sv[:len(uv)]
    canon = lambda a: np.where(np.isnan(a), np.nan, a)  # noqa: E731  (the text writer spells every NaN "NaN")
    for ext in ("bal", "bbal"):
        path = str(tmp_path / f"rt.{ext}")
        ba.write_gpu(path, ctx)
        rp = resident(c2b, ctx)
        st = rp.read(path)
        cams, p, g = download(c2b, rp, st)
        exp_p, exp_uv = (ba.points, ba.vis_graph.uv) if ext == "bbal" else (canon(ba.points), canon(ba.vis_graph.uv))
        assert bits_equal(p, exp_p), ext
        assert np.array_equal(g.offsets, ba.vis_graph.offsets) and np.array_equal(g.point_idx, ba.vis_graph.point_idx)
        assert bits_equal(g.uv.reshape(-1, 2), exp_uv), ext
        assert st["regrouped"] == 0


def from_vec_records(c2b, vecs):
    L, pd = c2b._lib.lib(), ctypes.POINTER(ctypes.c_double)
    out = np.zeros((len(vecs), 15))
    for i, v in enumerate(np.ascontiguousarray(vecs, np.float64)):
        L.c2b_camera_from_vec(v.ctypes.data_as(pd), out[i].ctypes.data_as(pd))
    return out


def file_vecs(path, ba_ref):
    """the camera 9-vectors as the file holds them"""
    C, O = ba_ref.num_cameras(), ba_ref.num_observations()
    if path.endswith(".bbal"):
        s = 24 + 8 * C + 24 * O
        return np.frombuffer(open(path, "rb").read()[s:s + 72 * C], ">f8").astype(np.float64).reshape(-1, 9)
    toks = open(path).read().split()
    return np.array(toks[3 + 4 * O:3 + 4 * O + 9 * C], np.float64).reshape(-1, 9)


def assert_same_as_mirror(c2b, ctx, path, what=""):
    ref = c2b.BAProblem.from_file(path)
    st = {}
    got = c2b.BAProblem.from_file_gpu(path, ctx, stats=st)
    assert np.array_equal(got.vis_graph.offsets, ref.vis_graph.offsets), what
    assert np.array_equal(got.vis_graph.point_idx, ref.vis_graph.point_idx), what
    assert bits_equal(got.vis_graph.uv, ref.vis_graph.uv), what
    assert bits_equal(got.points, ref.points), what
    assert bits_equal(got.cameras, from_vec_records(c2b, file_vecs(path, ref))), what
    ulp = np.abs(got.cameras.view(np.int64) - ref.cameras.view(np.int64))
    close = (ulp <= 2) | (np.abs(got.cameras - ref.cameras) <= 1e-300)
    assert close.all(), f"{what}: camera records more than 2 ulp from Python's from_vec"
    return got, st


def test_whole_files_against_mirrors(c2b, ctx, tmp_path):
    rng = np.random.default_rng(25)
    for C, P, k in [(1, 1, 3), (7, 40, 9), (60, 800, 50), (400, 20000, 300)]:
        ba = random_problem(c2b, rng, C, P, k, empty_every=5)
        for ext, write in (("bal", ba.write_text), ("bbal", ba.write_binary)):
            path = str(tmp_path / f"m{C}.{ext}")
            write(path)
            got, st = assert_same_as_mirror(c2b, ctx, path, f"C={C} {ext}")
            assert st["regrouped"] == 0 and st["n_obs"] == ba.num_observations()


@pytest.mark.parametrize("case", ["empty", "cameras_no_obs", "points_only"])
def test_edge_problems(c2b, ctx, tmp_path, case):
    rng = np.random.default_rng(26)
    ba = {"empty": lambda: random_problem(c2b, rng, 0, 0, 0),
          "cameras_no_obs": lambda: random_problem(c2b, rng, 6, 10, 0),
          "points_only": lambda: random_problem(c2b, rng, 0, 25, 0)}[case]()
    for ext in ("bal", "bbal"):
        path = str(tmp_path / f"e.{ext}")
        ba.write_gpu(path, ctx)
        got, _ = assert_same_as_mirror(c2b, ctx, path, f"{case} {ext}")
        assert (got.num_cameras(), got.num_points(), got.num_observations()) == \
            (ba.num_cameras(), ba.num_points(), ba.num_observations())


# ---- order and layout ------------------------------------------------------------------------------------------------
def text_parts(path):
    lines = open(path).read().split("\n")
    C, P, O = (int(t) for t in lines[0].split())
    return lines[0], lines[1:1 + O], lines[1 + O:1 + O + C + P]


def test_shuffled_observations_are_grouped(c2b, ctx, tmp_path):
    rng = np.random.default_rng(27)
    ba = random_problem(c2b, rng, 200, 3000, 60, empty_every=7)
    path = str(tmp_path / "s.bal")
    ba.write_text(path)
    head, obs, rest = text_parts(path)
    perm = rng.permutation(len(obs))
    with open(path, "w") as f:
        f.write("\n".join([head] + [obs[i] for i in perm] + rest) + "\n")
    got, st = assert_same_as_mirror(c2b, ctx, path, "shuffled")
    assert st["regrouped"] == 1
    # within a camera, file order: the shuffled lines of each camera in the order they now appear
    cam = np.array([int(obs[i].split()[0]) for i in perm])
    pt = np.array([int(obs[i].split()[1]) for i in perm])
    order = np.argsort(cam, kind="stable")
    assert np.array_equal(got.vis_graph.point_idx, pt[order])


def test_whitespace_layouts(c2b, ctx, tmp_path):
    rng = np.random.default_rng(28)
    ba = random_problem(c2b, rng, 30, 200, 20, empty_every=4)
    path = str(tmp_path / "ref.bal")
    ba.write_gpu(path, ctx)
    text = open(path).read()
    toks = text.split()
    variants = {
        "tabs": "\t".join(toks) + "\n",
        "crlf": text.replace("\n", "\r\n"),
        "runs": "   ".join(toks) + "  \n\n",
        "leading": " \n\t \r\n" + text,
        "no_final_newline": text.rstrip("\n"),
        "one_line": " ".join(toks),
        "vt_ff": "\v\f".join(toks),
        "trailing_garbage": text + "garbage 1.2.3 -x\n+++\n",
    }
    ref = c2b.BAProblem.from_file_gpu(path, ctx)
    for name, body in variants.items():
        p = str(tmp_path / f"{name}.bal")
        open(p, "w", newline="").write(body)
        got = c2b.BAProblem.from_file_gpu(p, ctx)
        assert np.array_equal(got.vis_graph.offsets, ref.vis_graph.offsets), name
        assert np.array_equal(got.vis_graph.point_idx, ref.vis_graph.point_idx), name
        assert bits_equal(got.vis_graph.uv, ref.vis_graph.uv), name
        assert bits_equal(got.points, ref.points) and bits_equal(got.cameras, ref.cameras), name


# ---- chunk boundaries ------------------------------------------------------------------------------------------------
def test_chunk_boundaries(c2b, ctx, tmp_path):
    rng = np.random.default_rng(29)
    ba = random_problem(c2b, rng, 40, 3000, 30, empty_every=3)
    ba.points[::7] = 5e-324  # 326-byte tokens
    paths = {ext: str(tmp_path / f"c.{ext}") for ext in ("bal", "bbal")}
    for p in paths.values():
        ba.write_gpu(p, ctx)
    ref = {ext: c2b.BAProblem.from_file_gpu(p, ctx) for ext, p in paths.items()}
    try:
        for chunk in (4096, 4104, 4096 + 24 * 7, 4096 + 24 * 100):
            ctx.tune("bal_chunk_bytes", chunk)
            for ext, p in paths.items():
                st = {}
                got = c2b.BAProblem.from_file_gpu(p, ctx, stats=st)
                assert st["chunks"] >= os.path.getsize(p) // chunk, (chunk, ext)
                r = ref[ext]
                assert np.array_equal(got.vis_graph.offsets, r.vis_graph.offsets), (chunk, ext)
                assert np.array_equal(got.vis_graph.point_idx, r.vis_graph.point_idx), (chunk, ext)
                assert bits_equal(got.vis_graph.uv, r.vis_graph.uv), (chunk, ext)
                assert bits_equal(got.points, r.points) and bits_equal(got.cameras, r.cameras), (chunk, ext)
        ctx.tune("bal_chunk_bytes", 4096)
        long_tok = str(tmp_path / "long.bal")
        open(long_tok, "w").write("0 1 0\n1." + "1" * 5000 + " 2 3\n")
        with pytest.raises(ParseError, match="byte 6"):
            c2b.BAProblem.from_file_gpu(long_tok, ctx)
    finally:
        ctx.tune("reset", 0)


# ---- malformed input -------------------------------------------------------------------------------------------------
GOOD = "2 3 2\n0 1 0.5 -0.5\n1 2 1e-3 7\n" + "0 0 0 1 2 3 500 0 0\n" * 2 + "1 2 3\n4 5 6\n7 8 9\n"


def text_cases():
    def at(s, old, new):
        i = GOOD.index(old)
        return GOOD[:i] + new + GOOD[i + len(old):], i
    c = {}
    c["bad_header"] = ("2 x 2" + GOOD[5:], 2)
    c["negative_header"] = ("-2" + GOOD[1:], 0)
    c["minus_index"] = at(GOOD, "1 2 1e-3", "-1 2 1e-3")
    c["fraction_index"] = at(GOOD, "0 1 0.5", "1.5 1 0.5")
    body, i = at(GOOD, "1 2 1e-3", "1 1e0 1e-3")
    c["exponent_index"] = (body, i + 2)
    c["u64_overflow_index"] = at(GOOD, "1 2 1e-3", "18446744073709551616 2 1e-3")
    c["u64_overflow_header"] = ("18446744073709551616" + GOOD[1:], 0)
    c["bad_number"] = at(GOOD, "500", "5O0")
    c["bad_number_2"] = at(GOOD, "7\n", "1e\n")
    c["nan_word"] = at(GOOD, "-0.5", "-nanx")
    return c


@pytest.mark.parametrize("case", list(text_cases()))
def test_malformed_text(c2b, ctx, tmp_path, case):
    body, off = text_cases()[case]
    path = str(tmp_path / "bad.bal")
    open(path, "w").write(body)
    good = str(tmp_path / "good.bal")
    open(good, "w").write(GOOD)
    rp = resident(c2b, ctx)
    rp.read(good)
    with pytest.raises(ParseError, match=f"byte {off}:"):
        rp.read(path)
    assert c2b._lib.lib().c2b_write_bal_resident(ctx.handle, str(tmp_path / "o.bal").encode(), 0, None) == INVALID
    if case != "u64_overflow_index":  # Python's int() takes any length: its mirror fails the range assert instead
        with pytest.raises(ParseError):
            c2b.BAProblem.from_file(path)  # the mirror agrees it is malformed


def test_malformed_sizes(c2b, ctx, tmp_path):
    rp = resident(c2b, ctx)
    lib = c2b._lib.lib()
    cases = {"too_few": GOOD.rsplit("7 8 9", 1)[0], "beyond_size": "1000 1000 1000\n0 0 1 1\n",
             "empty_file": "", "header_only": "1 1"}
    for name, body in cases.items():
        path = str(tmp_path / f"{name}.bal")
        open(path, "w").write(body)
        with pytest.raises(ParseError, match="byte"):
            rp.read(path)
        assert lib.c2b_write_bal_resident(ctx.handle, str(tmp_path / "o.bal").encode(), 0, None) == INVALID, name


def binary_file(ba, path):
    ba.write_binary(path)
    return bytearray(open(path, "rb").read())


def test_malformed_binary(c2b, ctx, tmp_path):
    rng = np.random.default_rng(30)
    ba = random_problem(c2b, rng, 5, 20, 6)
    ba.vis_graph.offsets[:] = [0, 3, 5, 9, 12, 14]
    ba.vis_graph.point_idx = ba.vis_graph.point_idx[:14] if len(ba.vis_graph.point_idx) >= 14 else \
        rng.integers(0, 20, 14).astype(np.uint64)
    ba.vis_graph.uv = rng.normal(size=(14, 2))
    good = binary_file(ba, str(tmp_path / "g.bbal"))
    rp = resident(c2b, ctx)
    lib = c2b._lib.lib()
    cases = {}
    cases["truncated_mid_record"] = good[:24 + 8 + 24 * 2 + 12]
    cases["truncated_mid_camera"] = good[:700]
    cases["truncated_points"] = good[:-4]
    b = bytearray(good)
    b[24:32] = struct.pack(">Q", 15)  # camera 0 claims more than the 14 observations
    cases["count_beyond_left"] = b
    b = bytearray(good)
    b[24 + 8 + 24 * 3:24 + 8 + 24 * 3 + 8] = struct.pack(">Q", 1)  # camera 1: 1 instead of 2
    cases["counts_do_not_sum"] = b + bytes(24)
    b = bytearray(good)
    b[0:8] = struct.pack(">Q", 10 ** 6)
    cases["header_beyond_size"] = b
    for name, body in cases.items():
        path = str(tmp_path / f"{name}.bbal")
        open(path, "wb").write(bytes(body))
        with pytest.raises(ParseError, match="byte"):
            rp.read(path)
        assert lib.c2b_write_bal_resident(ctx.handle, str(tmp_path / "o.bal").encode(), 0, None) == INVALID, name


def test_indices_out_of_range(c2b, ctx, tmp_path):
    rp = resident(c2b, ctx)
    lib = c2b._lib.lib()
    for name, body in {"camera": GOOD.replace("1 2 1e-3", "2 2 1e-3"),
                       "point": GOOD.replace("0 1 0.5", "0 3 0.5")}.items():
        path = str(tmp_path / f"{name}.bal")
        open(path, "w").write(body)
        with pytest.raises(AssertionError, match="out of range"):
            rp.read(path)
        with pytest.raises(AssertionError):
            c2b.BAProblem.from_file(path)
        assert lib.c2b_read_bal_resident(ctx.handle, path.encode(), 0, None) == INVALID
        assert lib.c2b_write_bal_resident(ctx.handle, str(tmp_path / "o.bal").encode(), 0, None) == INVALID
    rng = np.random.default_rng(31)
    ba = random_problem(c2b, rng, 3, 10, 4)
    ba.vis_graph = c2b.VisGraph(np.array([0, 2, 2, 5], np.uint64), np.array([1, 2, 3, 4, 5], np.uint64),
                                rng.normal(size=(5, 2)))
    b = binary_file(ba, str(tmp_path / "g.bbal"))
    first = 24 + 8 + 48 + 8 + 8  # camera 2's first record (camera 0: 2 records, camera 1: none)
    b[first:first + 8] = struct.pack(">Q", 10)
    path = str(tmp_path / "p.bbal")
    open(path, "wb").write(bytes(b))
    with pytest.raises(AssertionError):
        rp.read(path)
    assert lib.c2b_write_bal_resident(ctx.handle, str(tmp_path / "o.bal").encode(), 0, None) == INVALID


def test_missing_file_and_format(c2b, ctx, tmp_path):
    rp = resident(c2b, ctx)
    lib = c2b._lib.lib()
    open(str(tmp_path / "good.bal"), "w").write(GOOD)
    rp.read(str(tmp_path / "good.bal"))
    with pytest.raises(IOError_):
        rp.read(str(tmp_path / "missing.bal"))
    assert lib.c2b_write_bal_resident(ctx.handle, str(tmp_path / "o.bal").encode(), 0, None) == INVALID
    assert lib.c2b_read_bal_resident(ctx.handle, str(tmp_path / "good.bal").encode(), 7, None) == INVALID
    with pytest.raises(IOError_):
        rp.read(str(tmp_path / "good.txt"))


# ---- the resident chain ----------------------------------------------------------------------------------------------
def _visibility(c2b, ctx, n, cpb, ppb):
    from city2ba_b200 import synthetic
    cams = synthetic.grid_cameras(cpb, n, 20.0, 1.0)
    pts = synthetic.grid_points(ppb, n, 20.0, 1.0, 1.0)
    xyz, tri = synthetic.city_mesh(n)
    scene = c2b.Scene(xyz, tri, ctx=ctx)
    rp = resident(c2b, ctx)
    rp.upload_cameras(cams)
    rp.upload_points(pts)
    rp.run(scene, 10.0)
    st = rp.cull()
    c, p = rp.download_problem(st["n_cameras"], st["n_points"])
    return rp, c, p, rp.download()


def _chain(c2b, ctx, tmp_path, n, cpb, ppb, what):
    rp, cams, pts, g = _visibility(c2b, ctx, n, cpb, ppb)
    for ext in ("bal", "bbal"):
        path = str(tmp_path / f"chain.{ext}")
        rp.write(path)
        fresh = c2b.Context(0)
        try:
            r = resident(c2b, fresh)
            st = r.read(path)
            c2, p2, g2 = download(c2b, r, st)
            assert np.array_equal(g2.offsets, g.offsets) and np.array_equal(g2.point_idx, g.point_idx), what
            assert bits_equal(g2.uv, g.uv) and bits_equal(p2, pts), what
            assert bits_equal(c2, from_vec_records(c2b, camera_vecs(c2b, cams))), what
            host = c2b.BAProblem.from_file(path)
            # the C++ mirror's from_vec, bit for bit (Python's is within 2 ulp), so that the chains below match
            host.cameras = from_vec_records(c2b, file_vecs(path, host))
            for norm in (1.0, 2.0):
                assert r.reprojection_error(norm) == pytest.approx(host.total_reprojection_error(norm), rel=1e-12)
            # resident noise + write == from_file -> host-array noise entries -> write_gpu
            r.add_drift(0.01, 0.001, 0.1, seed=3)
            r.add_noise(0.01, 0.001, 0.01, 0.001, seed=4)
            out_r = str(tmp_path / f"noised_r.{ext}")
            r.write(out_r)
            from city2ba_b200 import noise
            h = noise.add_drift_normalized(host, 0.01, 0.001, 0.1, seed=3, ctx=fresh)
            h = noise.add_noise(h, 0.01, 0.001, 0.01, 0.001, seed=4, ctx=fresh)
            out_h = str(tmp_path / f"noised_h.{ext}")
            h.write_gpu(out_h, fresh)
            assert open(out_r, "rb").read() == open(out_h, "rb").read(), f"{what} {ext}: noise chain"
            # read -> resident cull -> write == from_file -> cull() -> write
            r.read(path)
            r.cull()
            out_c = str(tmp_path / f"culled_r.{ext}")
            r.write(out_c)
            out_hc = str(tmp_path / f"culled_h.{ext}")
            host = c2b.BAProblem.from_file(path)
            host.cameras = from_vec_records(c2b, file_vecs(path, host))
            host.cull().write_gpu(out_hc, fresh)
            assert open(out_c, "rb").read() == open(out_hc, "rb").read(), f"{what} {ext}: cull chain"
        finally:
            fresh.close()


def test_resident_chain_cfg2(c2b, ctx, tmp_path):
    _chain(c2b, ctx, tmp_path, 4, 10, 10, "cfg2")


def test_resident_chain_cfg3_full_size(c2b, ctx, tmp_path):
    _chain(c2b, ctx, tmp_path, 16, 9, 306, "cfg3")


# ---- the C++ mirror --------------------------------------------------------------------------------------------------
def test_cpp_read_on_gpu_equals_host(tmp_path):
    from test_bal_read_host import build_test_bal_read
    exe = build_test_bal_read(tmp_path)
    r = subprocess.run([exe, str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
