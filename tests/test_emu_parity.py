"""CPU: the kernel sources compiled for the host (tests/_emu, -DBATOTP_HOST_EMU: every kernel
body run sequentially, see batotp_b200/csrc/emu.h) against the oracle.  This checks the exact
per-thread program that runs on the B200 — and the chunk pipeline / C-ABI around it — without a
GPU; the `-m gpu` tests repeat it on the device."""
import hashlib

import numpy as np
import pytest

import _parity as P
from batotp_b200 import native


@pytest.fixture(scope="module")
def ctx():
    import __graft_entry__ as g
    c = native.Context(0, g.build_emu())
    # The library would pick the group-per-trajectory sweep kernel for batches this small; under the emulation its
    # many shuffles cost a fibre switch each, so the suite runs the one-trajectory-per-lane kernel unless a test
    # asks for the other one (test_group_sweep_kernel_*).
    c.set_sweep_kernel(1)
    yield c
    c.close()


@pytest.mark.parametrize("name", P.STOCK)
def test_stock_folders_reproduce_reference_files(ctx, name):
    cfg, tres, th, ca, ts = P.load_stock(name)
    res = P.run_device(ctx, cfg, tres, th, ca, ts)
    assert res.status[0] & native.ST_FATAL_MASK == 0
    d = P.GOLD + "/stock/" + name
    assert P.device_traj_out_bytes(cfg, res, 0) == open(d + "/ref_traj_out.dat", "rb").read()
    assert P.device_s_sdot_bytes(res, 0) == open(d + "/ref_s-sdot.dat", "rb").read()
    orc = P.OracleRun(cfg, tres, None if th is None else th[0], None if ca is None else ca[0],
                      None if ts is None else ts[0])
    assert P.compare(cfg, res, 0, orc) == []


@pytest.mark.parametrize("name,count", [("GEN7DOF", 24), ("KUKA", 2), ("CSPR3DOF", 3)])
def test_synthetic_batches_match_oracle_and_golden(ctx, name, count):
    g = P.synthetic_json()[name]
    cfg, tres, th, ca = P.load_synth(name, 0, count)
    res = P.run_device(ctx, cfg, tres, th, ca)
    for b in range(count):
        orc = P.OracleRun(cfg, tres, None if th is None else th[b], None if ca is None else ca[b])
        assert P.compare(cfg, res, b, orc) == [], b
        assert (res.n_rev[b], res.n_fwd[b], res.n_out[b]) == (g["n_rev"][b], g["n_fwd"][b], g["n_out"][b])
        assert hashlib.sha256(res.theta_out[b, :, :res.n_out[b]].tobytes()).hexdigest() == g["theta_out_sha256"][b]


def test_chunking_and_capacity_retries_do_not_change_results(ctx):
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 40, 10)
    ctx.set_chunk(4)  # 3 chunks: 4 + 4 + 2
    a = P.run_device(ctx, cfg, tres, th, None)
    ctx.set_chunk(16384)
    ctx.set_out_chunk(3)  # 4 output passes over the single resident chunk: 3 + 3 + 3 + 1
    b = P.run_device(ctx, cfg, tres, th, None)
    ctx.set_out_chunk(8192)
    c = P.run_device(ctx, cfg, tres, th, None)
    for nm in ("status", "n_rev", "n_fwd", "n_out", "t_total", "theta_out", "hist", "flags"):
        assert np.array_equal(getattr(a, nm), getattr(b, nm)), nm
        assert np.array_equal(getattr(a, nm), getattr(c, nm)), nm


def test_ragged_short_and_degenerate_inputs(ctx):
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 7, 6)
    th = th.copy()
    n0 = np.array([400, 57, 3, 2, 1, 400], dtype=np.int32)
    th[5, :, :] = th[5, :, :1]  # all points identical -> "no optimization" (ba.cpp:484-488)
    th[1, :, 20:25] = th[1, :, 19:20]  # repeated points -> remClosePts removes them (util.cpp:452)
    res = P.run_device(ctx, cfg, tres, th, None, n0=n0)
    for b in range(6):
        orc = P.OracleRun(cfg, tres, th[b], None, n0=int(n0[b]))
        assert P.compare(cfg, res, b, orc) == [], (b, res.status[b])
    assert res.status[4] & 1 and res.status[5] & (1 | 2)
    assert res.status[0] == 0 or res.status[0] == native.ST_BISECT_FAIL


def test_per_sample_mvc_matches_oracle(ctx):
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 3, 2)
    bi = ctx.make_in(th, None, tres)
    ctx.load(cfg, bi)
    ctx.interp_input()
    from _oracle import Oracle
    got = ctx.mvc_per_sample(2, 2048, 1.0e3)
    for b in range(2):
        o = Oracle(cfg)
        o.load_raw(400, tres, th[b])
        assert o.interp_input() == 0
        want = o.mvc_per_sample(1.0e3)
        assert np.array_equal(got[b, :len(want)], want)
        assert want.min() > 0 and want.max() < 1.0e3


def test_tail_overlap_does_not_change_results(ctx):
    """The last chunk of a batch runs on the library's second context, driven by its own host thread, when it fits
    one sweep CTA per SM (batotp_cuda_optimize_batch).  Under the emulation the launches of the two threads take
    turns, so this checks the hand-over logic: same outputs and same work counters with and without it.  A step
    hint below the steps of a tail path makes stragglers on both contexts: those of the second one are merged back
    and re-run with the others in one extra sweep pass."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 60, 11)
    ctx.set_chunk(4)  # 2 full chunks on the main context, 3 paths on the second one
    try:
        runs = []
        for on in (True, False, True):
            ctx.set_tail_overlap(on)
            ctx.stats_reset()
            r = P.run_device(ctx, cfg, tres, th, None)
            runs.append((r, ctx.stats()))
        ctx.set_step_hint(int(np.maximum(runs[1][0].n_rev, runs[1][0].n_fwd)[8:].max()) - 1)
        hinted = []
        for on in (True, False):
            ctx.set_tail_overlap(on)
            ctx.stats_reset()
            r = P.run_device(ctx, cfg, tres, th, None)
            hinted.append((r, ctx.stats()))
    finally:
        ctx.set_step_hint(0)
        ctx.set_tail_overlap(True)
        ctx.set_chunk(16384)
    (a, sa), (b, sb), (c, sc) = runs
    assert (a.status & native.ST_FATAL_MASK == 0).all()
    for nm in ("status", "n_rev", "n_fwd", "n_out", "t_total", "s_last_sec", "theta_out", "hist", "flags"):
        assert np.array_equal(getattr(a, nm), getattr(b, nm)), nm
        assert np.array_equal(getattr(a, nm), getattr(c, nm)), nm
        for r, _ in hinted:
            assert np.array_equal(getattr(r, nm), getattr(b, nm)), nm
    for k in ("verifies", "steps", "trajectories", "sweep_launches"):
        assert sa[k] == sb[k] == sc[k], k
    for _, sh in hinted:
        for k in ("verifies", "steps", "trajectories"):
            assert sh[k] == sb[k], k
        assert sh["sweep_launches"] == sb["sweep_launches"] + 1  # the stragglers' pass
    # (the launch totals may differ by a planning pass: the second context learns its capacities on first use)
    for bb in (0, 5, 9, 10):
        orc = P.OracleRun(cfg, tres, th[bb], None)
        assert P.compare(cfg, a, bb, orc) == [], bb


def test_sweep_filters_decide_nearly_everything(ctx):
    """The sweep kernel takes the bisection decisions from float models of the bounds (one common margin, then
    per-joint margins) and falls back to the exact quotients when neither separates.  Results are exact either way (checked above); this guards the speed path:
    the fallbacks must stay rare, otherwise the kernel silently degenerates into the all-exact one."""
    import ctypes as C
    out = (C.c_longlong * 16)()
    ctx.L.batotp_emu_filter_stats(out, 16, 1)
    cfg, tres, th, ca = P.load_synth("GEN7DOF", 100, 8)
    P.run_device(ctx, cfg, tres, th, ca)
    ctx.L.batotp_emu_filter_stats(out, 16, 1)
    certain, exact, b_joint, b_exact, v_skip, v_one, v_all = list(out)[:7]
    assert list(out)[8:11] == [0, 0, 0]  # every shortcut agreed with the full exact computation (TEST-ONLY blocks)
    assert certain > 100000
    assert exact < 0.01 * certain        # decisions deferred to the exact verification
    assert b_exact < 0.001 * b_joint     # bounds that needed all joints instead of the certified one
    assert v_all < 0.001 * (v_skip + v_one + 1)


@pytest.mark.parametrize("acc,vel,integ", [(0.05, 1.0, 1.0), (20.0, 0.2, 1.0), (1.0, 5.0, 1.0), (1.0, 1.0, 0.25),
                                           (300.0, 30.0, 0.5)])
def test_limit_regimes_match_oracle(ctx, acc, vel, integ):
    """The float models of the sweep kernel certify decisions relative to the size of the bounds they see, so the
    GEN7DOF paths are run with the limits and the step scaled far away from the stock values: acceleration-starved
    (every point bisects), velocity-bound, nearly unconstrained (the +-sddotmax clamp and the sdot cap come into
    play), and a fine step (larger clamp).  Everything must still equal the oracle bit for bit."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 900, 3)
    for i in range(cfg.n_joints):
        cfg.jnt_acc_max[i] *= acc
        cfg.jnt_vel_max[i] *= vel
    cfg.integ_res *= integ
    import ctypes as C
    st = (C.c_longlong * 16)()
    ctx.L.batotp_emu_filter_stats(st, 16, 1)
    res = P.run_device(ctx, cfg, tres, th, None, out_cap=65536, hist_cap=65536)
    ctx.L.batotp_emu_filter_stats(st, 16, 1)
    for b in range(3):
        orc = P.OracleRun(cfg, tres, th[b], None)
        assert P.compare(cfg, res, b, orc) == [], b
    # the host build cross-checks every shortcut against the full exact computation: decisions, settled bounds,
    # velocity caps (k_sweep.cuh, TEST-ONLY blocks)
    assert st[0] > 10000 and list(st)[8:11] == [0, 0, 0], list(st)


@pytest.mark.parametrize("ulps", [-2, 2])
def test_results_do_not_depend_on_the_float_reciprocal(ctx, ulps):
    """The floats of the sweep kernel only certify outcomes of the exact computation, so moving the approximate
    reciprocal they are built from by 2 units in the last place (rcp.approx on the device is good to 1) may change
    neither a single output bit nor a single cross-check."""
    import ctypes as C
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 1500, 4)
    for i in range(cfg.n_joints):
        cfg.jnt_acc_max[i] *= 0.3
    st = (C.c_longlong * 16)()
    ctx.L.batotp_emu_set_rcp_ulps(ulps)
    try:
        ctx.L.batotp_emu_filter_stats(st, 16, 1)
        res = P.run_device(ctx, cfg, tres, th, None, out_cap=65536, hist_cap=65536)
        ctx.L.batotp_emu_filter_stats(st, 16, 1)
    finally:
        ctx.L.batotp_emu_set_rcp_ulps(0)
    for b in range(4):
        orc = P.OracleRun(cfg, tres, th[b], None)
        assert P.compare(cfg, res, b, orc) == [], b
    assert st[0] > 10000 and list(st)[8:11] == [0, 0, 0], list(st)


def test_branch_free_bracket_update_equals_the_reference_shaped_one(ctx):
    """Bisect::step_any (one straight-line pass for every verification of the sweep kernel) against Bisect::step
    (the shape of ba.cpp:1270-1321) on random feasibility thresholds, including thresholds exactly at a
    candidate, zero / negative thresholds (bracket collapse, 100-pass limit) and non-positive start values."""
    assert ctx.selftest_bisect(12345, 400000) == 0


def test_step_capacity_is_bounded(ctx):
    """A trajectory that needs more Runge-Kutta steps than the configured ceiling keeps BATOTP_ST_STEP_CAP and
    is reported as not optimised; the batch call itself succeeds and the other trajectories are unaffected."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 7, 3)
    ref = P.run_device(ctx, cfg, tres, th, None)
    assert (ref.status & native.ST_FATAL_MASK == 0).all() and ref.n_fwd.min() > 1100
    ctx.set_max_steps(1024)
    try:
        c = native.Context(0, ctx.L._name)  # fresh capacities
        c.set_max_steps(1024)
        capped = P.run_device(c, cfg, tres, th, None)
        c.close()
    finally:
        ctx.set_max_steps(65536)
    assert ((capped.status & 32) != 0).all() and (capped.n_out == 0).all()
    again = P.run_device(ctx, cfg, tres, th, None)
    assert np.array_equal(again.theta_out, ref.theta_out) and np.array_equal(again.t_total, ref.t_total)


@pytest.mark.parametrize("name", ["RR", "UR5", "KUKA-LWR-IV", "CSPR3DOF"])
def test_automatic_integration_resolution(ctx, name):
    """SURVEY 8f rank 2: _isAutoIntegRes = true (per-trajectory integRes / weights, ba.cpp:471-556) against the
    oracle, which tests/test_oracle_vs_reference.py pins to the unmodified reference in this mode."""
    cfg, tres, th, ca, ts = P.load_stock(name)
    cfg = cfg.copy()
    cfg.is_auto_integ_res = 1
    res = P.run_device(ctx, cfg, tres, th, ca, ts)
    assert res.status[0] & native.ST_FATAL_MASK == 0
    orc = P.OracleRun(cfg, tres, None if th is None else th[0], None if ca is None else ca[0],
                      None if ts is None else ts[0])
    assert orc.ok and P.compare(cfg, res, 0, orc) == []


def test_interpolation_only_mode(ctx):
    """SURVEY 8f rank 2: _isInterpOnly (ba.cpp:139-159) — the path is only re-sampled at outRes.  UR5 carries
    joint and Cartesian rows (axis-angle -> quaternion -> axis-angle around the resample)."""
    from _oracle import Oracle
    cfg, tres, th, ca, ts = P.load_stock("UR5")
    cfg = cfg.copy()
    cfg.is_interp_only = 1
    res = P.run_device(ctx, cfg, tres, th, ca, ts, out_cap=8192)
    o = Oracle(cfg)
    o.load_raw(th.shape[2], tres, th[0], ca[0], None if ts is None else ts[0])
    assert o.interp_input() == -1
    n = int(o.scalar("nPts"))
    assert res.status[0] == 0 and res.n_out[0] == n and res.n_cart_out[0] == n and res.out_sres[0] == cfg.out_res
    assert np.array_equal(res.theta_out[0, :, :n], o.rows("theta", cfg.n_joints).astype(np.float32))
    assert np.array_equal(res.cart_out[0, :6, :n], o.rows("cart", 6).astype(np.float32))
    assert res.n_rev[0] == 0 and res.n_fwd[0] == 0 and not res.hist.any()
    # a batch of joint-only paths: absent Cartesian rows are zeros (the reference has no defined result there)
    cfg2, tres2, th2, _ = P.load_synth("GEN7DOF", 0, 5)
    cfg2 = cfg2.copy()
    cfg2.is_interp_only = 1
    r2 = P.run_device(ctx, cfg2, tres2, th2, None, out_cap=1024)
    assert (r2.status == 0).all() and (r2.n_out == r2.n_out[0]).all() and r2.n_out[0] > 400
    assert np.abs(r2.theta_out[:, :, 0] - th2[:, :, 0]).max() == 0  # a spline interpolates its first knot exactly


def test_batch_writer_files_are_the_reference_formats(ctx, tmp_path):
    """SURVEY 8f rank 1: the batch writer's traj_out_<i>.dat / s-sdot_<i>.dat are trajWriteBIN / sdotWrite
    byte for byte: the stock GEN7DOF folder gives the reference's own files, synthetic paths the packers that
    the golden files pin; a trajectory that was not optimised gets no file."""
    import os
    g = __import__("__graft_entry__")
    w = native.Writer(str(tmp_path), threads=3, lib_path=g.build_emu())
    cfg, tres, th, ca, ts = P.load_stock("GEN7DOF")
    res = P.run_device(ctx, cfg, tres, th, ca, ts)
    w.submit(cfg, res, 100, 0, 1)
    cfg2, tres2, th2, _ = P.load_synth("GEN7DOF", 20, 6)
    th2 = th2.copy()
    th2[3] = th2[3][:, :1]  # a path that does not move: not optimised
    res2 = P.run_device(ctx, cfg2, tres2, th2, None)
    assert res2.status[3] & native.ST_FATAL_MASK
    w.submit(cfg2, res2, 0, 0, 6)
    rc, written, failed = w.wait()
    w.close()
    assert (rc, written, failed) == (0, 6, 0)
    d = P.GOLD + "/stock/GEN7DOF"
    assert open(os.path.join(str(tmp_path), "traj_out_0000100.dat"), "rb").read() == open(d + "/ref_traj_out.dat", "rb").read()
    assert open(os.path.join(str(tmp_path), "s-sdot_0000100.dat"), "rb").read() == open(d + "/ref_s-sdot.dat", "rb").read()
    for b in range(6):
        f = os.path.join(str(tmp_path), "traj_out_%07d.dat" % b)
        if b == 3:
            assert not os.path.exists(f)
            continue
        assert open(f, "rb").read() == P.device_traj_out_bytes(cfg2, res2, b)
        assert open(os.path.join(str(tmp_path), "s-sdot_%07d.dat" % b), "rb").read() == P.device_s_sdot_bytes(res2, b)


def test_two_contexts_with_different_configs_do_not_disturb_each_other():
    """The run options travel with every launch (Ws is a kernel parameter), so contexts that hold different
    configurations can be driven phase by phase in any interleaving (round-1 advisor finding: a process-global
    config made context A compute with B's limits)."""
    import __graft_entry__ as g
    lib = g.build_emu()
    a, b = native.Context(0, lib), native.Context(0, lib)
    try:
        cfgA, tresA, thA, _ = P.load_synth("GEN7DOF", 0, 2)
        cfgB, tresB, thB, _ = P.load_synth("KUKA", 0, 1)
        a.load(cfgA, a.make_in(thA, None, tresA))
        a.interp_input()
        b.load(cfgB, b.make_in(thB, None, tresB))
        b.interp_input()
        a.sweeps()
        b.sweeps()
        a.interp_output()
        b.interp_output()
        ra = a.fetch(native.BatchResult(2, cfgA.n_joints, cfgA.n_cart, 8192, 8192, False))
        rb = b.fetch(native.BatchResult(1, cfgB.n_joints, cfgB.n_cart, 32768, 32768, False))
        for k in range(2):
            assert P.compare(cfgA, ra, k, P.OracleRun(cfgA, tresA, thA[k], None)) == []
        assert P.compare(cfgB, rb, 0, P.OracleRun(cfgB, tresB, thB[0], None)) == []
    finally:
        a.close()
        b.close()


def test_context_reuse_across_robots_and_path_lengths(ctx):
    """One context, robots with different row counts and path lengths one after the other: the input staging
    sets keep separate capacities for the joint and the Cartesian block (round-1 advisor finding: RR stock twice,
    then GEN7DOF, wrote past the staging buffer)."""
    for name in ("RR", "RR", "GEN7DOF", "CSPR3DOF", "UR5", "RR"):
        cfg, tres, th, ca, ts = P.load_stock(name)
        res = P.run_device(ctx, cfg, tres, th, ca, ts)
        d = P.GOLD + "/stock/" + name
        assert P.device_traj_out_bytes(cfg, res, 0) == open(d + "/ref_traj_out.dat", "rb").read(), name
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 0, 3)
    res = P.run_device(ctx, cfg, tres, th, None)
    assert P.compare(cfg, res, 2, P.OracleRun(cfg, tres, th[2], None)) == []


def test_phase_api_load_leaves_the_chunk_setting_alone(ctx):
    """batotp_cuda_load sizes the resident workspace from its own batch and must not turn the automatic
    chunking (0) into `chunk = B of the last phase-wise load` (round-1 advisor finding)."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 0, 5)
    ctx.set_chunk(0)
    ctx.load(cfg, ctx.make_in(th[:1], None, tres))
    ctx.interp_input()
    ctx.stats_reset()
    P.run_device(ctx, cfg, tres, th, None)
    assert ctx.stats()["sweep_launches"] == 1  # one chunk of 5, not five chunks of 1
    ctx.set_chunk(16384)


def test_stragglers_are_rerun_with_a_larger_step_capacity(ctx):
    """A few trajectories that outgrow the step capacity of their chunk do not make the whole chunk run again:
    they are re-run together after the batch (batotp_cuda.cu run_stragglers).  Same results as a run whose
    capacity served everybody; the sweep kernel is launched once per chunk plus once for the stragglers."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 100, 20)
    ctx.set_chunk(10)  # two chunks
    try:
        ctx.set_step_hint(0)
        a = P.run_device(ctx, cfg, tres, th, None)
        steps = np.sort(np.maximum(a.n_rev, a.n_fwd))
        hint = int(steps[-4])  # three trajectories need more steps than this capacity
        assert steps[-3] > hint >= steps[-5]
        ctx.set_step_hint(hint)
        ctx.stats_reset()
        b = P.run_device(ctx, cfg, tres, th, None)
        st = ctx.stats()
    finally:
        ctx.set_step_hint(0)
        ctx.set_chunk(16384)
    assert (b.status & native.ST_FATAL_MASK == 0).all()
    for nm in ("status", "n_rev", "n_fwd", "n_out", "n_grid", "t_total", "t_rev", "s_last_sec", "out_sres",
               "theta_out", "hist", "flags"):
        assert np.array_equal(getattr(a, nm), getattr(b, nm)), nm
    assert st["sweep_launches"] == 3 and st["trajectories"] == 20


def test_results_into_device_resident_buffers(ctx):
    """batotp_batch_out.on_device: every pointer of the result is device memory (here, under the emulation, plain
    memory): scalars arrive through k_fetch_scalars, rows through the same packed staging sets."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 30, 7)
    ctx.set_chunk(4)
    ctx.set_out_chunk(3)
    try:
        a = P.run_device(ctx, cfg, tres, th, None, out_cap=4096, hist_cap=4096)
        b = native.BatchResult(7, cfg.n_joints, cfg.n_cart, 4096, 4096, False)
        b.c.on_device = 1
        ctx.optimize_batch(cfg, ctx.make_in(th, None, tres), b)
    finally:
        ctx.set_chunk(16384)
        ctx.set_out_chunk(8192)
    for nm in ("status", "n_rev", "n_fwd", "n_out", "n_cart_out", "n_grid", "t_total", "t_rev", "s_last_sec",
               "out_sres", "theta_out", "hist", "flags"):
        assert np.array_equal(getattr(a, nm), getattr(b, nm)), nm


@pytest.mark.parametrize("name,decim,window", [("GEN7DOF", 3, 1), ("GEN7DOF", 2, 4), ("RR", 3, 3), ("UR5", 1, 3),
                                               ("UR5", 3, 3), ("CSPR3DOF", 3, 3), ("KUKA-LWR-IV", 2, 4)])
def test_input_decimation_and_smoothing(ctx, name, decim, window, tmp_path):
    """inputDecimFact / smoothWindow (ba.cpp:195-242, quirk Q6) on the device: k_in_smooth_decimate + k_in_decim_fix
    against the oracle (which tests/test_oracle_vs_reference.py pins to the unmodified reference for these options)."""
    cfg, tres, th, ca, ts = P.load_stock_variant(name, tmp_path, inputDecimFact=decim, smoothWindow=window)
    res = P.run_device(ctx, cfg, tres, th, ca, ts)
    orc = P.OracleRun(cfg, tres, None if th is None else th[0], None if ca is None else ca[0],
                      None if ts is None else ts[0])
    assert orc.ok and res.status[0] & native.ST_FATAL_MASK == 0
    assert P.compare(cfg, res, 0, orc) == []


def test_strict_trig_port_reproduces_the_host_libm(ctx):
    """cfg.trig_mode 1: sin / cos of the point functions are a port of the host libm's algorithm (k_trig.cuh).
    The host build of the same functions against this machine's libm, in the arithmetic glibc selected here;
    the other arithmetic is checked in a child process started with glibc's FMA variants switched off."""
    import os
    import subprocess
    import sys
    bad, variant = ctx.selftest_trig(2026, 3_000_000)
    assert bad == 0 and variant in (1, 3)
    code = ("import sys; sys.path.insert(0, %r); import __graft_entry__ as g; from batotp_b200 import native; "
            "c = native.Context(0, g.build_emu()); print(c.selftest_trig(11, 1500000))" % P.HERE.rsplit("/", 1)[0])
    env = dict(os.environ, GLIBC_TUNABLES="glibc.cpu.hwcaps=-FMA,-AVX2", BATOTP_TRIG_VARIANT="1")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.strip().splitlines()[-1] == "(0, 1)"
    if variant == 3:  # the check bites: the fused port against the unfused libm differs
        env["BATOTP_TRIG_VARIANT"] = "3"
        out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
        assert out.returncode == 0 and out.stdout.strip().splitlines()[-1] != "(0, 3)"


@pytest.mark.parametrize("name", ["RR", "KUKA-LWR-IV", "UR5"])
def test_host_evaluated_trig_mode_gives_the_same_bytes(ctx, name):
    """trig_mode 2 (the host evaluates the trig-bearing point functions with its libm between device stages) and
    trig_mode 1 (the device port) are both strict: same files as the reference."""
    cfg, tres, th, ca, ts = P.load_stock(name)
    d = P.GOLD + "/stock/" + name
    for mode in (1, 2):
        c2 = cfg.copy()
        c2.trig_mode = mode
        res = P.run_device(ctx, c2, tres, th, ca, ts)
        assert P.device_traj_out_bytes(c2, res, 0) == open(d + "/ref_traj_out.dat", "rb").read(), mode
        assert P.device_s_sdot_bytes(res, 0) == open(d + "/ref_s-sdot.dat", "rb").read(), mode


@pytest.mark.parametrize("name", ["GEN7DOF", "RR", "UR5", "CSPR3DOF"])
def test_group_sweep_kernel_on_stock_folders(ctx, name):
    """k_sweep_group.cuh (a group of 8 / 4 lanes per trajectory, per-joint work spread over the lanes, shuffle
    reductions) gives the reference's files byte for byte, like the one-trajectory-per-lane kernel: joint limits
    only (GEN7DOF), serial torque + Cartesian (RR, 4 lanes), Cartesian with quaternions (UR5), Par2Ser torque (CSPR)."""
    cfg, tres, th, ca, ts = P.load_stock(name)
    ctx.set_sweep_kernel(2)
    try:
        res = P.run_device(ctx, cfg, tres, th, ca, ts)
    finally:
        ctx.set_sweep_kernel(1)
    d = P.GOLD + "/stock/" + name
    assert P.device_traj_out_bytes(cfg, res, 0) == open(d + "/ref_traj_out.dat", "rb").read()
    assert P.device_s_sdot_bytes(res, 0) == open(d + "/ref_s-sdot.dat", "rb").read()
    orc = P.OracleRun(cfg, tres, None if th is None else th[0], None if ca is None else ca[0],
                      None if ts is None else ts[0])
    assert P.compare(cfg, res, 0, orc) == []  # switching flags and sLastSec included


def test_group_sweep_kernel_on_a_ragged_batch(ctx):
    """Several groups per warp, trajectories of different lengths, refills from the queue, a degenerate path."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 300, 9)
    th = th.copy()
    n0 = np.array([400, 400, 57, 400, 3, 400, 1, 400, 400], dtype=np.int32)
    ctx.set_sweep_kernel(1)
    a = P.run_device(ctx, cfg, tres, th, None, n0=n0, out_cap=4096, hist_cap=4096)
    ctx.set_sweep_kernel(2)
    try:
        ctx.stats_reset()
        b = P.run_device(ctx, cfg, tres, th, None, n0=n0, out_cap=4096, hist_cap=4096)
        sb = ctx.stats()
    finally:
        ctx.set_sweep_kernel(1)
    for nm in ("status", "n_rev", "n_fwd", "n_out", "t_total", "s_last_sec", "theta_out", "hist", "flags"):
        assert np.array_equal(getattr(a, nm), getattr(b, nm)), nm
    assert sb["verifies"] > 0 and P.compare(cfg, b, 3, P.OracleRun(cfg, tres, th[3], None)) == []


def test_chunks_shrink_until_the_workspace_fits(ctx, monkeypatch):
    """A chunk whose workspace would not fit the device memory is refused before anything is allocated, with the
    size that fits; the batch goes on with smaller chunks and gives the same results.  When even one trajectory
    does not fit the call fails with a message instead of retrying for ever.  (BATOTP_EMU_FREE_MB makes the host
    emulation report that much free memory; 2 GB of it are the planner's own reserve.)"""
    import __graft_entry__ as g
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 0, 12)
    a = P.run_device(ctx, cfg, tres, th, None, out_cap=4096, hist_cap=4096)
    fresh = native.Context(0, g.build_emu())  # no workspace yet: every size is planned against the "free" memory
    fresh.set_sweep_kernel(1)
    try:
        monkeypatch.setenv("BATOTP_EMU_FREE_MB", str(2048 + 8))  # room for a few trajectories
        b = P.run_device(fresh, cfg, tres, th, None, out_cap=4096, hist_cap=4096)
        n1 = fresh.stats()["sweep_launches"]
        assert n1 >= 3
        for nm in ("status", "n_rev", "n_fwd", "n_out", "t_total", "theta_out", "hist", "flags"):
            assert np.array_equal(getattr(a, nm), getattr(b, nm)), nm
        # the next call of the same configuration starts with the chunk size that fitted (no refused attempt, the
        # workspace of the first call is reused as it is)
        fresh.stats_reset()
        b2 = P.run_device(fresh, cfg, tres, th, None, out_cap=4096, hist_cap=4096)
        assert fresh.stats()["sweep_launches"] <= n1 and np.array_equal(b2.theta_out, a.theta_out)
        cfg2, tres2, th2, ca2, ts2 = P.load_stock("KUKA-LWR-IV")  # another robot: the workspace is planned anew
        monkeypatch.setenv("BATOTP_EMU_FREE_MB", "2048")
        with pytest.raises(native.NativeError, match="of workspace"):
            P.run_device(fresh, cfg2, tres2, th2, ca2, ts2)
        monkeypatch.delenv("BATOTP_EMU_FREE_MB")
        c = P.run_device(fresh, cfg, tres, th, None, out_cap=4096, hist_cap=4096)
        assert np.array_equal(a.theta_out, c.theta_out)
    finally:
        fresh.close()


@pytest.mark.parametrize("name", ["RR", "UR5", "CSPR3DOF", "KUKA-LWR-IV"])
def test_per_sample_mvc_on_cartesian_and_torque_robots(ctx, name):
    """SURVEY 8a A10 on robots with Cartesian limits (UR5, KUKA), serial torque (RR) and Par2Ser torque (CSPR3DOF):
    k_mvc against the oracle, which tests/test_oracle_vs_reference.py pins to the reference's private per-point
    functions on the same folders."""
    from _oracle import Oracle
    cfg, tres, th, ca, ts = P.load_stock(name)
    ctx.load(cfg, ctx.make_in(th, ca, tres, timestamp=ts))
    ctx.interp_input()
    o = Oracle(cfg)
    n0 = (th if th is not None else ca).shape[2]
    o.load_raw(n0, tres, None if th is None else th[0], None if ca is None else ca[0], None if ts is None else ts[0])
    assert o.interp_input() == 0
    for start in (1.0e3, 0.5):
        want = o.mvc_per_sample(start)
        got = ctx.mvc_per_sample(1, len(want) + 8, start)
        assert np.array_equal(got[0, :len(want)], want), start


def _kuka_torque_cfg(cfg):
    """The KUKA torque variant of SURVEY 8d C3: the stock KUKA options plus torque limits on a caller-supplied model."""
    c = cfg.copy()
    c.is_trq_on = 1
    c.dyn_source = 1
    for j, v in enumerate((60.0, 60.0, 30.0, 30.0, 15.0, 15.0, 8.0)):
        c.jnt_trq_max[j] = v
        c.jnt_trq_min[j] = -v
    return c


def test_caller_supplied_dynamics(ctx):
    """cfg.dyn_source = 1 (batotp_cuda_set_dyn_callback): (a) dynRR behind the plug-in signature gives the reference's
    RR files byte for byte; (b) the KUKA-LWR-IV stock path with torque limits on a 7-joint model the reference does
    not have (k_sweep<7,true,true>): same host point function on both sides, device against the oracle bit for bit
    - switching flags, torque rows and all - with the limits actually binding."""
    from _oracle import dyn_fn_address
    cfg, tres, th, ca, ts = P.load_stock("RR")
    c1 = cfg.copy()
    c1.dyn_source = 1
    try:
        ctx.set_dyn_callback(dyn_fn_address("orc_demo_dyn_rr"))
        res = P.run_device(ctx, c1, tres, th, ca, ts)
        d = P.GOLD + "/stock/RR"
        assert P.device_traj_out_bytes(c1, res, 0) == open(d + "/ref_traj_out.dat", "rb").read()
        assert P.device_s_sdot_bytes(res, 0) == open(d + "/ref_s-sdot.dat", "rb").read()
        cfg, tres, th, ca, ts = P.load_stock("KUKA-LWR-IV")
        plain = P.run_device(ctx, cfg, tres, th, ca, ts)
        c2 = _kuka_torque_cfg(cfg)
        fn = dyn_fn_address("orc_demo_dyn_serial")
        ctx.set_dyn_callback(fn)
        res = P.run_device(ctx, c2, tres, th, ca, ts)
        orc = P.OracleRun(c2, tres, th[0], None, dyn_fn=fn)
        assert orc.ok and res.status[0] & native.ST_FATAL_MASK == 0
        assert P.compare(c2, res, 0, orc) == []
        assert res.t_total[0] > plain.t_total[0]  # the torque limits bind: the move takes longer
    finally:
        ctx.set_dyn_callback(None)
    c3 = _kuka_torque_cfg(cfg)
    with pytest.raises(native.NativeError, match="dyn_source = 1 needs a point function"):
        P.run_device(ctx, c3, tres, th, ca, ts)


def test_ragged_rows_hold_the_same_samples(ctx):
    """batotp_batch_out.row_offset: joint rows packed at their own length ([J][n_out] blocks, the payload of
    trajWriteBIN) instead of the pitch of the longest trajectory - same float32 samples as the pitched layout, blocks
    disjoint and inside the capacity, also across chunks, output sub-chunks, the tail helper and re-run stragglers."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 400, 21)
    a = P.run_device(ctx, cfg, tres, th, None, out_cap=4096, hist_cap=64)
    total = int(a.n_out.sum())
    steps = np.sort(np.maximum(a.n_rev, a.n_fwd))
    ctx.set_chunk(8)
    ctx.set_out_chunk(3)
    try:
        for hint in (0, int(steps[-3])):
            ctx.set_step_hint(hint)
            b = native.BatchResult(21, cfg.n_joints, cfg.n_cart, 0, 0, False, want_hist=False, ragged_cap=total + 5)
            ctx.optimize_batch(cfg, ctx.make_in(th, None, tres), b)
            assert np.array_equal(a.n_out, b.n_out) and np.array_equal(a.t_total, b.t_total)
            spans = sorted((int(b.row_offset[k]), int(b.row_offset[k]) + int(b.n_out[k])) for k in range(21))
            assert spans[0][0] >= 0 and spans[-1][1] <= total and all(x[1] <= y[0] for x, y in zip(spans, spans[1:]))
            for k in range(21):
                assert np.array_equal(b.rows(k), a.theta_out[k, :, :a.n_out[k]]), k
        small = native.BatchResult(21, cfg.n_joints, cfg.n_cart, 0, 0, False, want_hist=False, ragged_cap=total // 2)
        with pytest.raises(native.NativeError, match="ragged_cap"):
            ctx.optimize_batch(cfg, ctx.make_in(th, None, tres), small)
    finally:
        ctx.set_step_hint(0)
        ctx.set_chunk(16384)
        ctx.set_out_chunk(8192)
    # torque rows travel the same way (RR: serial torque)
    cfg, tres, th, ca, ts = P.load_stock("RR")
    p = P.run_device(ctx, cfg, tres, th, ca, ts)
    r = native.BatchResult(1, cfg.n_joints, cfg.n_cart, 0, 0, True, want_hist=False, ragged_cap=4096)
    ctx.optimize_batch(cfg, ctx.make_in(th, ca, tres, timestamp=ts), r)
    n = int(p.n_out[0])
    assert np.array_equal(r.rows(0), p.theta_out[0, :, :n]) and np.array_equal(r.rows(0, "trq_out"), p.trq_out[0, :, :n])


def test_parallel_torque_without_par2ser(ctx, tmp_path):
    """SURVEY 8f rank 3: cable-tension limits of the CSPR3DOF with isPar2Ser = 0 (ba.cpp:1463-1491: the structure
    matrix is rebuilt at every point and every verification solves 2 x 3 three-by-three systems with a replaced
    column) - k_sweep<3,true,true,PAR> against the oracle, which tests/test_oracle_vs_reference.py pins to the
    unmodified reference for this option."""
    cfg, tres, th, ca, ts = P.load_stock_variant("CSPR3DOF", tmp_path, isPar2Ser=0)
    assert cfg.is_par2ser == 0
    res = P.run_device(ctx, cfg, tres, th, ca, ts)
    orc = P.OracleRun(cfg, tres, None, ca[0])
    assert orc.ok and res.status[0] & native.ST_FATAL_MASK == 0
    assert P.compare(cfg, res, 0, orc) == []
    cfg2, tres2, _, ca2 = P.load_synth("CSPR3DOF", 50, 3)
    cfg2 = cfg2.copy()
    cfg2.is_par2ser = 0
    r2 = P.run_device(ctx, cfg2, tres2, None, ca2)
    for b in range(3):
        assert P.compare(cfg2, r2, b, P.OracleRun(cfg2, tres2, None, ca2[b])) == [], b


def test_max_integration_time_is_reported_like_the_reference(ctx):
    """maxIntegTime (ba.cpp:1117-1122): a sweep that does not reach the end of the path within maxIntegTime/integRes
    steps ends with BA::MAX_INTEGRATION_TIME in the reference (sweep returns -1); here the trajectory gets
    BATOTP_ST_MAX_INTEG_TIME (not the internal step ceiling) and no output, the rest of the batch is untouched."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 900, 4)
    ref = P.run_device(ctx, cfg, tres, th, None)
    c2 = cfg.copy()
    c2.max_integ_time = 0.6 * float(ref.t_total.min())  # every path needs longer than this
    res = P.run_device(ctx, c2, tres, th, None)
    assert ((res.status & 16) != 0).all() and ((res.status & 32) == 0).all() and (res.n_out == 0).all()
    for b in range(2):
        orc = P.OracleRun(c2, tres, th[b], None)
        assert not orc.ok
    c3 = cfg.copy()
    c3.max_integ_time = 0.5 * (float(np.sort(ref.t_total)[1]) + float(np.sort(ref.t_total)[2]))  # two of the four finish
    mix = P.run_device(ctx, c3, tres, th, None)
    done = (mix.status & native.ST_FATAL_MASK) == 0
    assert 1 <= done.sum() <= 3
    for b in range(4):
        orc = P.OracleRun(c3, tres, th[b], None)
        assert orc.ok == bool(done[b]), b
        if done[b]:
            assert P.compare(c3, mix, b, orc) == [], b


@pytest.mark.parametrize("name", P.STOCK)
def test_walker_kernels_give_the_same_bytes(ctx, name):
    """The sequential walkers of interpInputData exist in two shapes: one thread per trajectory (k_adjust_s forming the
    norm increments itself, k_march) for chunks that fill the device, and point-parallel increments (k_adjust_inc) + a
    group of 16 lanes per trajectory (k_march_group: one coordinate row per lane, the squared differences summed in the
    reference's order from shuffled values) for small chunks.  Every stock robot through both, byte for byte the
    reference's files - incl. the Cartesian rows that are only carried along (Traj::cartpt) and the UR5's 13 rows."""
    cfg, tres, th, ca, ts = P.load_stock(name)
    d = P.GOLD + "/stock/" + name
    out = []
    for mode in (1, 2):
        ctx.set_walker_kernel(mode)
        try:
            res = P.run_device(ctx, cfg, tres, th, ca, ts)
        finally:
            ctx.set_walker_kernel(0)
        assert P.device_traj_out_bytes(cfg, res, 0) == open(d + "/ref_traj_out.dat", "rb").read(), mode
        assert P.device_s_sdot_bytes(res, 0) == open(d + "/ref_s-sdot.dat", "rb").read(), mode
        out.append(res)
    assert np.array_equal(out[0].n_grid, out[1].n_grid)


def test_walker_kernels_on_a_ragged_batch(ctx):
    """Two groups per warp with trajectories of different lengths (the groups of a warp diverge), degenerate paths
    (fewer than 4 points after the march: the linear stretch to 4 points), automatic integration resolution."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 700, 9)
    n0 = np.array([400, 400, 57, 400, 3, 400, 1, 400, 400], dtype=np.int32)
    runs = []
    for auto in (0, 1):
        cfg.is_auto_integ_res = auto
        for mode in (1, 2):
            ctx.set_walker_kernel(mode)
            try:
                runs.append(P.run_device(ctx, cfg, tres, th, None, n0=n0, out_cap=8192, hist_cap=8192))
            finally:
                ctx.set_walker_kernel(0)
        a, b = runs[-2:]
        for nm in ("status", "n_rev", "n_fwd", "n_out", "n_grid", "t_total", "s_last_sec", "theta_out", "hist", "flags"):
            assert np.array_equal(getattr(a, nm), getattr(b, nm)), (auto, nm)
    cfg.is_auto_integ_res = 0
    assert P.compare(cfg, runs[1], 3, P.OracleRun(cfg, tres, th[3], None)) == []


def test_chunks_are_cut_to_whole_sweep_rounds(ctx, monkeypatch):
    """A sweep launch lasts whole rounds of the trajectories it keeps resident, so once the occupancy of the
    configuration's sweep kernel is known (from its first launch) chunks of more than one round are cut to whole
    rounds (CSPR3DOF on the B200: memory allows 19072 paths per chunk, two rounds hold 18944).  TEST-ONLY knob:
    BATOTP_EMU_SWEEP_CAP makes the emulated launches report an occupancy of 10 trajectories (21 paths: the third round would be less than a quarter full)."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 2000, 21)
    a = P.run_device(ctx, cfg, tres, th, None)
    ctx.set_chunk(0)  # automatic chunking (an explicit chunk setting is taken literally)
    monkeypatch.setenv("BATOTP_EMU_SWEEP_CAP", "10")
    P.run_device(ctx, cfg, tres, th, None)  # learns the occupancy: 21 paths in one chunk
    ctx.stats_reset()
    b = P.run_device(ctx, cfg, tres, th, None)  # 20 + 1: the third round would hold 1 of 10
    st = ctx.stats()
    monkeypatch.delenv("BATOTP_EMU_SWEEP_CAP")
    assert st["sweep_launches"] == 2 and st["trajectories"] == 21
    for nm in ("status", "n_rev", "n_fwd", "n_out", "t_total", "s_last_sec", "theta_out", "hist", "flags"):
        assert np.array_equal(getattr(a, nm), getattr(b, nm)), nm
    other, tres2, th2, ca2, ts2 = P.load_stock("RR")  # another configuration forgets what was learnt
    P.run_device(ctx, other, tres2, th2, ca2, ts2)
    ctx.stats_reset()
    c = P.run_device(ctx, cfg, tres, th, None)
    assert ctx.stats()["sweep_launches"] == 1 and np.array_equal(c.theta_out, a.theta_out)
    ctx.set_chunk(16384)
