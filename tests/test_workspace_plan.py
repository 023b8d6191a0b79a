"""CPU (host emulation): the workspace planner counts exactly what a context allocates.

Before a chunk's arrays are allocated, the planner checks that they fit the free device memory beside a reserve for
the output arrays of one sub-chunk; a chunk that would not fit is refused with the size that would (from the bytes per
trajectory).  Both footprints are the allocation lists themselves, summed.  For the chunk arrays the planned and held
bytes therefore agree by construction (the same walk on both sides); what these tests pin is the output reserve - the
sub-chunk size, the output capacities derived from the step capacity, the pitches in use, the FP64 side output and the
fused path must be the ones the output arrays are then allocated for - and the per-trajectory figure.  Every case runs
on a fresh context, so that nothing held from an earlier request (the workspaces are reused when they cover a request)
enters the comparison."""
import ctypes as C

import pytest

import _parity as P
from batotp_b200 import native

# chunk arrays that do not grow with the trajectories: the sweep kernel's work-queue counter (4 int) and the closing
# entry of the ragged-layout offsets (1 long long)
FIXED_CHUNK_BYTES = 4 * 4 + 8


def _fresh():
    import __graft_entry__ as g
    c = native.Context(0, g.build_emu())
    c.set_sweep_kernel(1)  # the lane kernel: the group kernel's shuffles are slow under the emulation
    return c


@pytest.fixture
def ctx():
    c = _fresh()
    yield c
    c.close()


def _result(cfg, B, layout):
    trq = bool(cfg.is_trq_on)
    if layout == "pitched":  # the caller's pitches, larger than the device capacities
        return native.BatchResult(B, cfg.n_joints, cfg.n_cart, 32768, 16384, trq)
    if layout == "capacities":  # no rows or histories asked for: the staging sets at the device capacities
        return native.BatchResult(B, cfg.n_joints, cfg.n_cart, 0, 0, trq, want_rows=False, want_hist=False)
    return native.BatchResult(B, cfg.n_joints, cfg.n_cart, 0, 4096, trq, ragged_cap=B * 65536)


def _plan(ctx, cfg, tres, th, ca, ts=None, layout="pitched"):
    """Runs one batch; -> the planner's {chunk, out, perTraj} and the held {wsBytes, outBytes, B}."""
    B = (th if th is not None else ca).shape[0]
    res = _result(cfg, B, layout)
    ctx.optimize_batch(cfg, ctx.make_in(th, ca, tres, timestamp=ts), res)
    assert (res.status & native.ST_FATAL_MASK == 0).all(), res.status
    v = (C.c_size_t * 6)()
    assert ctx.L.batotp_emu_workspace_plan(ctx.h, v) == 0
    plan = dict(zip(("chunk", "out", "per_traj", "ws_bytes", "out_bytes", "B"), v))
    assert plan["B"] == B and plan["ws_bytes"] > 0 and plan["out_bytes"] > 0
    assert plan["chunk"] == plan["per_traj"] * B + FIXED_CHUNK_BYTES
    return plan


def _check(plan):
    assert (plan["chunk"], plan["out"]) == (plan["ws_bytes"], plan["out_bytes"])


# GEN7DOF: joint-only rows (R = J), output smoothing on the fused path.  KUKA-LWR-IV: Cartesian rows.  UR5: 7
# Cartesian rows (axis-angle in, quaternion inside).  RR and CSPR3DOF: torque limits, unfused output path.
@pytest.mark.parametrize("name", ["GEN7DOF", "KUKA-LWR-IV", "UR5", "RR", "CSPR3DOF"])
@pytest.mark.parametrize("layout", ["pitched", "capacities"])
def test_planned_footprints_equal_the_allocations(ctx, name, layout):
    cfg, tres, th, ca, ts = P.load_stock(name)
    _check(_plan(ctx, cfg, tres, th, ca, ts, layout))


@pytest.mark.parametrize("name", ["GEN7DOF", "RR"])
def test_planned_footprints_with_ragged_results(ctx, name):
    cfg, tres, th, ca, ts = P.load_stock(name)
    _check(_plan(ctx, cfg, tres, th, ca, ts, "ragged"))


def test_planned_footprints_with_fp64_side_output(ctx):
    cfg, tres, th, ca, ts = P.load_stock("GEN7DOF")
    ctx.set_keep_f64(True)
    with_f64 = _plan(ctx, cfg, tres, th, ca, ts)
    plain = _fresh()
    try:
        without = _plan(plain, cfg, tres, th, ca, ts)
    finally:
        plain.close()
    assert with_f64["out_bytes"] > without["out_bytes"]  # the FP64 rows are held ...
    _check(with_f64)  # ... and planned


def test_planned_footprints_over_several_sub_chunks(ctx):
    """A chunk of 6 paths leaves in output sub-chunks of 4 + 2: the output arrays are allocated for the first (and
    largest) one and serve the last one as they are, which is what the planner reserves (min(B, out chunk) paths)."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 0, 6)
    ctx.set_out_chunk(4)
    plan = _plan(ctx, cfg, tres, th, None)
    _check(plan)
    one_sub_chunk = _fresh()  # the same 6 paths in one output sub-chunk hold more
    try:
        assert _plan(one_sub_chunk, cfg, tres, th, None)["out_bytes"] > plan["out_bytes"]
    finally:
        one_sub_chunk.close()
