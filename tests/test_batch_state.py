"""CPU (host emulation): what a batch call (batotp_cuda_optimize_batch) keeps for itself.

The state of one batch call - the result layout, the straggler list, the tail hand-over - belongs to that call.  The
tail chunk it hands to the second context runs under the caller's settings, and nothing of the call is left on the
context for the phase-wise entry points (load, interp_input, sweeps, interp_output, fetch) that follow it."""
import numpy as np
import pytest

import _parity as P
from batotp_b200 import native

ST_STEP_CAP = 32  # BATOTP_ST_STEP_CAP
RESULTS = ("status", "n_rev", "n_fwd", "n_out", "n_cart_out", "n_grid", "t_total", "t_rev", "s_last_sec", "out_sres",
           "theta_out", "hist", "flags")


def _context():
    import __graft_entry__ as g
    c = native.Context(0, g.build_emu())
    c.set_sweep_kernel(1)  # the lane kernel: the group kernel's shuffles are slow under the emulation
    return c


@pytest.fixture(scope="module")
def ctx():
    c = _context()
    yield c
    c.close()


def test_tail_helper_runs_under_the_callers_settings(ctx):
    """44 paths in chunks of 16: two full chunks on the main context and a tail of 12 on the second one.  Every fourth
    path is short (150 points, under 1024 steps), the others take about 2000 steps.  The step hint starts each chunk
    at 1024 steps; more than eight paths of a chunk outgrow it, which is too many to re-run as stragglers, and doubling
    the capacity would pass the ceiling of 2047: the long paths keep BATOTP_ST_STEP_CAP.  A second context that fell
    back to the default ceiling (65536) would double its capacity and optimise the long tail paths."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 0, 44)
    n0 = np.where(np.arange(44) % 4 == 3, 150, th.shape[2]).astype(np.int32)
    ctx.set_chunk(16)
    ctx.set_max_steps(2047)
    ctx.set_step_hint(1024)
    ctx.set_walker_kernel(2)
    ctx.set_keep_f64(True)
    try:
        runs = []
        for on in (True, False):
            ctx.set_tail_overlap(on)
            ctx.stats_reset()
            r = P.run_device(ctx, cfg, tres, th, None, n0=n0, out_cap=4096, hist_cap=4096)
            runs.append((r, ctx.stats()))
    finally:
        ctx.set_tail_overlap(True)
        ctx.set_keep_f64(False)
        ctx.set_walker_kernel(0)
        ctx.set_step_hint(0)
        ctx.set_max_steps(65536)
        ctx.set_chunk(16384)
    (a, sa), (b, sb) = runs
    tail = a.status[32:]
    assert (tail & ST_STEP_CAP).any() and ((tail & native.ST_FATAL_MASK) == 0).any(), tail
    for nm in RESULTS:
        assert np.array_equal(getattr(a, nm), getattr(b, nm)), nm
    for k in ("verifies", "steps", "trajectories", "sweep_launches"):
        assert sa[k] == sb[k], k
    for k in (3, 35, 43):  # short paths, one of them on each side of the hand-over
        assert P.compare(cfg, a, k, P.OracleRun(cfg, tres, th[k], None, n0=int(n0[k]))) == [], k


def _phase_run(c, cfg, tres, th):
    c.load(cfg, c.make_in(th, None, tres))
    c.interp_input()
    c.sweeps()
    c.interp_output()
    return c.fetch(native.BatchResult(th.shape[0], cfg.n_joints, cfg.n_cart, 4096, 4096, False))


def test_batch_call_leaves_nothing_for_the_phase_api(ctx):
    """A ragged batch call with stragglers (two chunks of 10, a step hint three paths outgrow) and then a phase-wise
    run on the same context: the phase-wise rows are packed at the device capacities, pitched, and no straggler is
    collected - the same bytes as the phase-wise run on a fresh context."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 100, 20)
    ctx.set_chunk(10)
    try:
        ctx.set_step_hint(0)
        a = P.run_device(ctx, cfg, tres, th, None)
        steps = np.sort(np.maximum(a.n_rev, a.n_fwd))
        ctx.set_step_hint(int(steps[-4]))
        ctx.stats_reset()
        rag = native.BatchResult(20, cfg.n_joints, cfg.n_cart, 0, 0, False, want_hist=False,
                                 ragged_cap=int(a.n_out.sum()))
        ctx.optimize_batch(cfg, ctx.make_in(th, None, tres), rag)
        assert ctx.stats()["sweep_launches"] == 3  # two chunks and the stragglers' pass
        assert np.array_equal(rag.n_out, a.n_out)
    finally:
        ctx.set_step_hint(0)
        ctx.set_chunk(16384)
    got = _phase_run(ctx, cfg, tres, th[:6])
    fresh = _context()
    try:
        want = _phase_run(fresh, cfg, tres, th[:6])
    finally:
        fresh.close()
    assert (want.status & native.ST_FATAL_MASK == 0).all()
    for nm in RESULTS:
        assert np.array_equal(getattr(got, nm), getattr(want, nm)), nm
