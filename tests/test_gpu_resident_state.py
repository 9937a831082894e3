"""The entries that work on the resident problem's graph (c2b_cull_problem_resident,
c2b_add_incorrect_correspondences_resident, c2b_write_bal_resident) after each sequence of calls that leaves the
resident CSR in a different state: refused with the generic message when there is no graph, refused with the
host-buffer message while the CSR is the last camera batch of a host-buffer c2b_visibility_graph (also after resident
noise passes that move the points), accepted on the graph of a resident pass or of a resident cull."""
import ctypes
import os

import pytest

from city2ba_b200.baproblem import ParseError

pytestmark = pytest.mark.gpu

OK, INVALID = 0, -1
MAX_DIST = 10.0


def _problem():
    from city2ba_b200 import synthetic
    return synthetic.grid_cameras(10, 4, 20.0, 1.0), synthetic.grid_points(10, 4, 20.0, 1.0, 1.0)


def _host_call(c2b, rp, tmp_path):
    cams, pts = _problem()
    c2b.visibility_graph(None, cams, pts, MAX_DIST, occlusion="analytic", ctx=rp.ctx)


def _resident_graph(c2b, rp, tmp_path):
    cams, pts = _problem()
    rp.upload_cameras(cams)
    rp.upload_points(pts)
    rp.run(None, MAX_DIST, occlusion="analytic")


def _failed_read(c2b, rp, tmp_path):
    _resident_graph(c2b, rp, tmp_path)
    bad = str(tmp_path / "bad.bal")
    open(bad, "w").write("1 1")
    with pytest.raises(ParseError):
        rp.read(bad)


GENERIC, HOST_BUFFER = "no resident result", "host-buffer"

# state: (calls on a fresh ctx, expected status, phrase of the refusal)
STATES = {
    "fresh_ctx": (lambda c2b, rp, tmp_path: None, INVALID, GENERIC),
    "host_buffer_call": (_host_call, INVALID, HOST_BUFFER),
    "host_buffer_call_then_drift": (
        lambda c2b, rp, tmp_path: (_host_call(c2b, rp, tmp_path), rp.add_drift(0.01, 0.001, 0.1, seed=3)),
        INVALID, HOST_BUFFER),
    "host_buffer_call_then_sin_noise": (
        lambda c2b, rp, tmp_path: (_host_call(c2b, rp, tmp_path), rp.add_sin_noise([1, 0, 0], [0, 1, 0], 0.1, 1.0)),
        INVALID, HOST_BUFFER),
    "host_buffer_call_then_point_noise": (
        lambda c2b, rp, tmp_path: (_host_call(c2b, rp, tmp_path), rp.add_noise(0.01, 0.001, 0.01, 0.0, seed=4)),
        INVALID, HOST_BUFFER),
    "resident_graph": (_resident_graph, OK, None),
    "after_resident_cull": (lambda c2b, rp, tmp_path: (_resident_graph(c2b, rp, tmp_path), rp.cull()), OK, None),
    "after_failed_read": (_failed_read, INVALID, GENERIC),
}


def _cull(c2b, ctx, tmp_path):
    return c2b._lib.lib().c2b_cull_problem_resident(ctx.handle, ctypes.byref(c2b._lib.CullStats()))


def _mismatch(c2b, ctx, tmp_path):
    st = c2b._lib.MismatchStats()
    return c2b._lib.lib().c2b_add_incorrect_correspondences_resident(ctx.handle, 0.5, 1, ctypes.byref(st))


def _write(c2b, ctx, tmp_path):
    path = str(tmp_path / "out.bal")
    rc = c2b._lib.lib().c2b_write_bal_resident(ctx.handle, path.encode(), 0, None)
    assert os.path.exists(path) == (rc == OK)
    return rc


ENTRIES = {"cull": _cull, "mismatch": _mismatch, "write_bal": _write}


@pytest.mark.parametrize("state", list(STATES))
@pytest.mark.parametrize("entry", list(ENTRIES))
def test_graph_entries_by_resident_state(c2b, tmp_path, entry, state):
    setup, want, phrase = STATES[state]
    fresh = c2b.Context(0)
    try:
        setup(c2b, c2b.generate.ResidentProblem(fresh), tmp_path)
        rc = ENTRIES[entry](c2b, fresh, tmp_path)
        msg = c2b._lib.lib().c2b_last_error().decode()
        assert rc == want, msg
        if phrase:
            assert phrase in msg
    finally:
        fresh.close()
