"""The FP64 stages of the device path against the oracle, bit for bit (CPU: the host emulation of the kernels;
-m gpu: the product library on the device).

The other parity tests compare rows and histories after the cast to float32.  A wrong last bit in the sweep
usually changes a step count, so they notice it; a wrong last bit in the output phase feeds nothing back and
survives the cast unless it crosses a float32 rounding boundary.  The FP64 rows are a product of their own
(batotp_cuda_get_f64, the BATOTP::BA facade's Traj rows).  So here the device is driven phase by phase with the
FP64 side output on (batotp_cuda_set_keep_f64) next to one oracle per path, and after every phase the FP64
arrays are compared as uint64 bit patterns (-0 / +0 and NaN payloads count).  The cases reach every kernel
variant of the output phase: the smoothing windows of the fused evaluate-smooth-decimate kernels, the 6- and
7-joint row kernels, a BOTH path, the unfused smoothing of the torque and kinematics robots, re-interpolation,
windows that reach both ends of short paths, and both float32 packing kernels."""
import numpy as np
import pytest

import _parity as P
from _oracle import Oracle, dyn_fn_address
from batotp_b200 import native
from batotp_b200.config import BOTH

GPU = pytest.mark.gpu


@pytest.fixture(scope="module", params=["emu", pytest.param("gpu", marks=GPU)])
def ctx(request):
    """A context with the FP64 side output on: the host emulation of the kernels with the lane sweep kernel (the
    group kernel's shuffles are slow under the emulation), or the product library on the device with the
    library's own choice of kernels unless a test sets one."""
    import __graft_entry__ as g
    if request.param == "emu":
        c = native.Context(0, g.build_emu())
        c.set_sweep_kernel(1)
    else:
        if native.load().batotp_cuda_device_count() < 1:
            pytest.skip("no CUDA device")
        c = native.Context(0)
    c.kind = request.param
    c.set_keep_f64(True)
    yield c
    c.close()


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _diff(tag, got, want):
    """None when `got` holds the bit patterns of `want`, else the first differing index and the largest relative
    difference."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    if got.shape != want.shape:
        return "%s: %d values, oracle %d" % (tag, got.size, want.size)
    bad = np.flatnonzero(_bits(got) != _bits(want))
    if bad.size == 0:
        return None
    i = bad[0]
    with np.errstate(all="ignore"):
        rel = np.abs(got[bad] - want[bad]) / np.maximum(np.abs(want[bad]), np.finfo(np.float64).tiny)
    rel = np.where(np.isnan(rel), np.inf, rel)
    return "%s: %d of %d values differ, first at %d: %r, oracle %r; max relative difference %.3g" % (
        tag, bad.size, got.size, i, got[i], want[i], rel.max())


class _Check:
    """Collects the mismatches of one path (`where` prefixes every message)."""

    def __init__(self, ctx, b, where, msgs):
        self.ctx, self.b, self.where, self.msgs = ctx, b, where, msgs

    def rows(self, dev, o, orc_name, n, first=None):
        for r in range(n):
            try:
                got = self.ctx.get_f64(dev, self.b, r)
            except KeyError:
                self.msgs.append("%s %s[%d]: not held by the device" % (self.where, dev, r))
                continue
            want = o.vec(orc_name, r)
            if first is not None:
                if len(got) != first + 1:
                    self.msgs.append("%s %s[%d]: %d values, %d grid points" % (self.where, dev, r, len(got), first + 1))
                    continue
                got, want = got[:first], want[:first]
            m = _diff("%s %s[%d]" % (self.where, dev, r), got, want)
            if m:
                self.msgs.append(m)

    def vec(self, dev, want):
        m = _diff("%s %s" % (self.where, dev), self.ctx.get_f64(dev, self.b), want)
        if m:
            self.msgs.append(m)


def lockstep(ctx, cfg, tres, th, ca=None, ts=None, n0=None, dyn_fn=None):
    """Runs the batch through the device phases (load, interp_input, sweeps, interp_output) and one oracle per path
    (interp_input, sweep(-1, 0), sweep(1, 1), interp_output) in lock-step and compares the FP64 arrays after each
    phase.  Returns (mismatch messages, the fetched float32 result).  A path the oracle does not optimise must end
    with a fatal device status, and one it optimises with none."""
    ref = th if th is not None else ca
    B, n0max = ref.shape[0], ref.shape[2]
    lens = [n0max] * B if n0 is None else [int(x) for x in n0]
    J = cfg.n_joints
    msgs = []
    if dyn_fn is not None:
        ctx.set_dyn_callback(dyn_fn)
    try:
        ctx.load(cfg, ctx.make_in(th, ca, tres, n0=n0, timestamp=ts))
        ctx.interp_input()
        orcs, ok = [], []
        for b in range(B):
            n = lens[b]
            o = Oracle(cfg)
            if dyn_fn is not None:
                o.set_dyn_callback(dyn_fn)
            o.load_raw(n, tres, None if th is None else np.ascontiguousarray(th[b, :, :n]),
                       None if ca is None else np.ascontiguousarray(ca[b, :, :n]),
                       None if ts is None else ts[b, :n])
            rc = o.interp_input()
            orcs.append(o)
            chk = _Check(ctx, b, "path %d, interp_input:" % b, msgs)
            if cfg.is_interp_only:
                # the path is only re-sampled at outRes (ba.cpp:139-159): the oracle stops here with its rows ready
                ok.append(rc == -1)
                chk.rows("theta_out", o, "theta", J)
                chk.rows("cart_out", o, "cart", int(o.scalar("nCart")))
                continue
            ok.append(rc == 0 and o.scalar("nPts") >= 4)  # orc_optimize's two early exits
            if not ok[b]:
                continue
            chk.vec("integ_res", [o.scalar("integRes")])  # the automatic integRes is chosen here (ba.cpp:493-556)
            nC = int(o.scalar("nPtsC"))
            # The oracle's *C_y is the segment coefficient c0 of the spline, one per segment: its last entry is not a
            # knot (0, or for RR left over from an earlier spline), so only the nPtsC - 1 segment values are compared.
            chk.rows("thetaC_y", o, "thetaC_y", J, first=nC - 1)
            chk.rows("thetaC_m", o, "thetaC_m", J)
            nCart = int(o.scalar("nCart"))
            chk.rows("cartC_y", o, "cartC_y", nCart, first=nC - 1)
            chk.rows("cartC_m", o, "cartC_m", nCart)
            if cfg.is_trq_on:
                chk.rows("theta", o, "theta", J)
                chk.rows("cart", o, "cart", nCart)
                for k in "1234":
                    chk.rows("a" + k, o, "a" + k, J)
                    chk.rows("a%sC_m" % k, o, "a%sC_m" % k, J)
        if not cfg.is_interp_only:
            ctx.sweeps()
            for b in range(B):
                if not ok[b]:
                    continue
                o = orcs[b]
                ok[b] = o.sweep(-1, 0) == 0 and o.sweep(1, 1) == 0
                if not ok[b]:
                    continue
                chk = _Check(ctx, b, "path %d, sweeps:" % b, msgs)
                for dev, orc_name in (("s_rev", "hist_s0"), ("sdot_rev", "hist_sdot0"), ("s_fwd", "hist_s1"),
                                      ("sdot_fwd", "hist_sdot1")):
                    chk.vec(dev, o.vec(orc_name))
                for dev, orc_name in (("t_total", "tFwd"), ("t_rev", "tRev"), ("integ_res", "integRes")):
                    chk.vec(dev, [o.scalar(orc_name)])
            ctx.interp_output()
            for b in range(B):
                if not ok[b]:
                    continue
                o = orcs[b]
                assert o.interp_output() == 0
                chk = _Check(ctx, b, "path %d, interp_output:" % b, msgs)
                chk.rows("theta_out", o, "theta", J)
                chk.rows("cart_out", o, "cart", int(o.scalar("cartRows")))  # UR5: the axis-angle rows included
                if cfg.is_trq_on:
                    chk.rows("trq_out", o, "trq", J)
        res = ctx.fetch(native.BatchResult(B, J, cfg.n_cart, 0, 0, bool(cfg.is_trq_on), want_rows=False,
                                           want_hist=False))
    finally:
        if dyn_fn is not None:
            ctx.set_dyn_callback(None)
    for b in range(B):
        fatal = bool(res.status[b] & native.ST_FATAL_MASK)
        if fatal == ok[b]:
            msgs.append("path %d: device status %d, oracle %s" % (b, res.status[b], "ok" if ok[b] else "failed"))
        elif ok[b] and res.n_out[b] != int(orcs[b].scalar("nPts")):
            msgs.append("path %d: %d output points, oracle %d" % (b, res.n_out[b], int(orcs[b].scalar("nPts"))))
    return msgs, res


def _no_mismatch(msgs):
    assert not msgs, "%d FP64 mismatches:\n%s" % (len(msgs), "\n".join(msgs[:25]))


# ---------------------------------------------------------------------------------------------- stock robots

_KERNELS = [pytest.param("emu", 1, w, id="emu-lane-walker%d" % w) for w in (1, 2)] + [
    pytest.param("gpu", s, w, marks=GPU, id="gpu-%s-walker%d" % ("lane" if s == 1 else "group", w))
    for s in (1, 2) for w in (1, 2)]


@pytest.mark.parametrize("ctx,sweep,walker", _KERNELS, indirect=["ctx"])
@pytest.mark.parametrize("name", P.STOCK)
def test_stock_robots_stage_by_stage(ctx, sweep, walker, name):
    cfg, tres, th, ca, ts = P.load_stock(name)
    ctx.set_sweep_kernel(sweep)
    ctx.set_walker_kernel(walker)
    try:
        msgs, res = lockstep(ctx, cfg, tres, th, ca, ts)
    finally:
        ctx.set_sweep_kernel(1 if ctx.kind == "emu" else 0)
        ctx.set_walker_kernel(0)
    assert res.status[0] & native.ST_FATAL_MASK == 0
    _no_mismatch(msgs)


@pytest.mark.parametrize("name", P.STOCK)
@pytest.mark.parametrize("fact", [1, 2, 3, 4, 6, 7, 9, 11, 13])
def test_output_smoothing_windows(ctx, name, fact, tmp_path):
    """outSmoothFact picks the output kernel: the fused evaluate-smooth-decimate kernels of a joint path, one
    instantiation per window half-width (2..11 -> 1..5, the generic branch beyond; GEN7DOF's half-width 2 takes the
    7-row kernel), and the separate smoothing of the torque robots (RR, CSPR3DOF: Trq -> Trq2 too) and of the
    robots with output kinematics (KUKA-LWR-IV, UR5)."""
    cfg, tres, th, ca, ts = P.load_stock_variant(name, tmp_path, outSmoothFact=fact)
    assert cfg.out_smooth_fact == fact
    msgs, res = lockstep(ctx, cfg, tres, th, ca, ts)
    assert res.status[0] & native.ST_FATAL_MASK == 0
    _no_mismatch(msgs)


@pytest.mark.parametrize("out_res", [0.004, 0.01, 0.02])
@pytest.mark.parametrize("fact", [3, 5, 7, 9])
def test_output_resolution_and_smoothing(ctx, out_res, fact):
    """A synthetic GEN7DOF path (integRes 0.01): outRes 0.004 re-interpolates the smoothed rows (and scales the
    window, ba.cpp:1711-1716), 0.01 and 0.02 do not."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 11, 1)
    cfg = cfg.copy()
    cfg.out_smooth_fact = fact
    cfg.out_res = out_res
    msgs, res = lockstep(ctx, cfg, tres, th)
    assert res.status[0] & native.ST_FATAL_MASK == 0
    _no_mismatch(msgs)


@pytest.mark.parametrize("fact", [3, 5, 7])
def test_six_joint_generic_robot(ctx, fact):
    """n_joints = 6 on the GEN7DOF configuration: rows 0..5, the 6-row kernel at window 5."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 11, 2)
    cfg = cfg.copy()
    cfg.n_joints = 6
    cfg.out_smooth_fact = fact
    msgs, res = lockstep(ctx, cfg, tres, np.ascontiguousarray(th[:, :6]))
    assert (res.status & native.ST_FATAL_MASK == 0).all()
    _no_mismatch(msgs)


@pytest.mark.parametrize("fact", [3, 5, 9])
def test_both_path_with_smoothing(ctx, fact):
    """A generic BOTH path carries its Cartesian rows: the per-row fused kernel instead of the joint-row ones."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 11, 2)
    cfg = cfg.copy()
    cfg.path_type = BOTH
    cfg.out_smooth_fact = fact
    ca = np.ascontiguousarray(np.stack([0.3 * np.sin(th[:, 0]), 0.2 * np.cos(th[:, 1]), 0.1 * th[:, 2]], axis=1))
    msgs, res = lockstep(ctx, cfg, tres, th, ca)
    assert (res.status & native.ST_FATAL_MASK == 0).all()
    _no_mismatch(msgs)


@pytest.mark.parametrize("n0", [4, 6, 12])
@pytest.mark.parametrize("fact", [5, 11])
def test_short_paths_with_wide_windows(ctx, n0, fact):
    """Few output points against wide smoothing windows: the window reaches both ends of the rows (the shrinking
    end windows of smooth(), util.cpp:261-263).  The device's guard against a window wider than the rows
    (k_out_smooth_plan, BATOTP_ST_UNSUPPORTED) must not refuse a path the oracle smooths: the status has to agree."""
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 11, 1)
    cfg = cfg.copy()
    cfg.out_smooth_fact = fact
    msgs, _ = lockstep(ctx, cfg, tres, np.ascontiguousarray(th[:, :, :n0]))
    _no_mismatch(msgs)


# ---------------------------------------------------------------------------------------------- other options

@pytest.mark.parametrize("name", P.STOCK)
def test_automatic_integration_resolution(ctx, name):
    cfg, tres, th, ca, ts = P.load_stock(name)
    cfg = cfg.copy()
    cfg.is_auto_integ_res = 1
    msgs, res = lockstep(ctx, cfg, tres, th, ca, ts)
    # the automatic integRes of the GEN7DOF stock path is NaN in the reference's arithmetic (compared above as a
    # bit pattern): neither side optimises it
    assert bool(res.status[0] & native.ST_FATAL_MASK) == (name == "GEN7DOF")
    _no_mismatch(msgs)


@pytest.mark.parametrize("name,decim,window", [("GEN7DOF", 3, 1), ("GEN7DOF", 2, 4), ("RR", 3, 3), ("UR5", 1, 3),
                                               ("UR5", 3, 3), ("CSPR3DOF", 3, 3), ("KUKA-LWR-IV", 2, 4)])
def test_input_decimation_and_smoothing(ctx, name, decim, window, tmp_path):
    cfg, tres, th, ca, ts = P.load_stock_variant(name, tmp_path, inputDecimFact=decim, smoothWindow=window)
    msgs, res = lockstep(ctx, cfg, tres, th, ca, ts)
    assert res.status[0] & native.ST_FATAL_MASK == 0
    _no_mismatch(msgs)


def test_parallel_torque_without_par2ser(ctx, tmp_path):
    cfg, tres, th, ca, ts = P.load_stock_variant("CSPR3DOF", tmp_path, isPar2Ser=0)
    assert cfg.is_par2ser == 0
    msgs, res = lockstep(ctx, cfg, tres, th, ca, ts)
    assert res.status[0] & native.ST_FATAL_MASK == 0
    _no_mismatch(msgs)


def test_caller_supplied_dynamics(ctx):
    """dyn_source = 1: RR with the reference's dynamics behind the plug-in signature, and KUKA-LWR-IV with torque
    limits on a 7-joint model; the same host function feeds the device and the oracle."""
    cfg, tres, th, ca, ts = P.load_stock("RR")
    cfg = cfg.copy()
    cfg.dyn_source = 1
    msgs, res = lockstep(ctx, cfg, tres, th, ca, ts, dyn_fn=dyn_fn_address("orc_demo_dyn_rr"))
    assert res.status[0] & native.ST_FATAL_MASK == 0
    _no_mismatch(msgs)
    cfg, tres, th, ca, ts = P.load_stock("KUKA-LWR-IV")
    cfg = cfg.copy()
    cfg.is_trq_on = 1
    cfg.dyn_source = 1
    for j, v in enumerate((60.0, 60.0, 30.0, 30.0, 15.0, 15.0, 8.0)):
        cfg.jnt_trq_max[j] = v
        cfg.jnt_trq_min[j] = -v
    msgs, res = lockstep(ctx, cfg, tres, th, ca, ts, dyn_fn=dyn_fn_address("orc_demo_dyn_serial"))
    assert res.status[0] & native.ST_FATAL_MASK == 0
    _no_mismatch(msgs)


def test_interpolation_only_mode(ctx):
    """isInterpOnly on UR5: joint rows and the axis-angle rows re-sampled at outRes, nothing optimised."""
    cfg, tres, th, ca, ts = P.load_stock("UR5")
    cfg = cfg.copy()
    cfg.is_interp_only = 1
    msgs, res = lockstep(ctx, cfg, tres, th, ca, ts)
    assert res.status[0] == 0
    _no_mismatch(msgs)


# ---------------------------------------------------------------------------------------------- batches

def _batch_check(ctx, cfg, res, b, orc, msgs):
    """FP64 rows and histories of path b of an optimize_batch result (its output sub-chunk still held) against
    the oracle, and its float32 result."""
    msgs += ["path %d: %s" % (b, m) for m in P.compare(cfg, res, b, orc)]
    if not orc.ok:
        return
    o = orc.o
    chk = _Check(ctx, b, "path %d:" % b, msgs)
    for dev, orc_name in (("s_rev", "hist_s0"), ("sdot_rev", "hist_sdot0"), ("s_fwd", "hist_s1"),
                          ("sdot_fwd", "hist_sdot1")):
        chk.vec(dev, o.vec(orc_name))
    for dev, orc_name in (("t_total", "tFwd"), ("t_rev", "tRev"), ("integ_res", "integRes")):
        chk.vec(dev, [o.scalar(orc_name)])
    chk.rows("theta_out", o, "theta", cfg.n_joints)
    chk.rows("cart_out", o, "cart", int(o.scalar("cartRows")))
    if cfg.is_trq_on:
        chk.rows("trq_out", o, "trq", cfg.n_joints)


@pytest.mark.parametrize("ctx", [pytest.param("gpu", marks=GPU)], indirect=True)
@pytest.mark.parametrize("sweep", [1, 2], ids=["lane_kernel", "group_kernel"])
@pytest.mark.parametrize("name,count", [("GEN7DOF", 512), ("KUKA", 8), ("CSPR3DOF", 32)])
def test_batch_in_one_output_sub_chunk(ctx, name, count, sweep):
    """Every path of a batch in one chunk and one output sub-chunk (the FP64 side output holds the last
    sub-chunk only): FP64 rows and histories of every path against the oracle.  The step hint covers every path,
    so none is re-run as a straggler after the chunk."""
    cfg, tres, th, ca = P.load_synth(name, 0, count)
    orcs = [P.OracleRun(cfg, tres, None if th is None else th[b], None if ca is None else ca[b]) for b in range(count)]
    ctx.set_sweep_kernel(sweep)
    ctx.set_chunk(count)
    ctx.set_out_chunk(count)
    steps = max(max(o.n_rev, o.n_fwd) for o in orcs)  # KUKA: over 21 000 steps and output points
    ctx.set_step_hint(steps + 64)
    try:
        res = P.run_device(ctx, cfg, tres, th, ca, out_cap=max(o.n_out for o in orcs), hist_cap=steps)
    finally:
        ctx.set_step_hint(0)
        ctx.set_chunk(0)
        ctx.set_out_chunk(8192)
        ctx.set_sweep_kernel(0)
    msgs = []
    for b in range(count):
        _batch_check(ctx, cfg, res, b, orcs[b], msgs)
    assert all(o.ok for o in orcs)
    _no_mismatch(msgs)


def test_fp64_rows_of_a_path_outside_the_held_sub_chunk_are_refused(ctx):
    """With several output sub-chunks the FP64 rows of the last one are held: a path of an earlier sub-chunk gets
    KeyError, not the rows of whichever path now sits at its place; its histories stay (chunk-resident)."""
    B, sub = (512, 200) if ctx.kind == "gpu" else (9, 4)
    held = (B - 1) // sub * sub  # first path of the last sub-chunk
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 0, B)
    orcs = {b: P.OracleRun(cfg, tres, th[b], None) for b in (0, sub - 1, sub, held - 1, held, B - 1)}
    steps = P.run_device(ctx, cfg, tres, th, None, out_cap=8192, hist_cap=8192)
    ctx.set_chunk(B)
    ctx.set_out_chunk(sub)
    ctx.set_step_hint(int(np.maximum(steps.n_rev, steps.n_fwd).max()) + 64)  # no path is re-run as a straggler
    try:
        res = P.run_device(ctx, cfg, tres, th, None, out_cap=8192, hist_cap=8192)
    finally:
        ctx.set_step_hint(0)
        ctx.set_chunk(0)
        ctx.set_out_chunk(8192)
    msgs = []
    for b, orc in orcs.items():
        if b >= held:
            _batch_check(ctx, cfg, res, b, orc, msgs)
            continue
        for nm in ("theta_out", "cart_out"):
            with pytest.raises(KeyError):
                ctx.get_f64(nm, b, 0)
        chk = _Check(ctx, b, "path %d:" % b, msgs)
        chk.vec("s_fwd", orc.o.vec("hist_s1"))
        msgs += ["path %d: %s" % (b, m) for m in P.compare(cfg, res, b, orc)]
    _no_mismatch(msgs)


@pytest.mark.parametrize("ragged", [False, True], ids=["pitched", "ragged"])
def test_pack_kernels_give_the_same_float_rows(ctx, ragged):
    """Without the FP64 side output a generic joint robot's float32 rows are packed by k_out_pack_rows (warp tiles
    through shared memory), with it by k_out_pack: rows, histories, flags and scalars must be the same bytes."""
    B = 512 if ctx.kind == "gpu" else 12
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 0, B)
    runs = []
    try:
        for keep in (False, True):
            ctx.set_keep_f64(keep)
            if ragged:
                r = native.BatchResult(B, cfg.n_joints, cfg.n_cart, 0, 4096, False, ragged_cap=B * 4096)
                ctx.optimize_batch(cfg, ctx.make_in(th, None, tres), r)
            else:
                r = P.run_device(ctx, cfg, tres, th, None, out_cap=4096, hist_cap=4096)
            runs.append(r)
    finally:
        ctx.set_keep_f64(True)
    a, b = runs
    assert (a.status & native.ST_FATAL_MASK == 0).all()
    assert a.n_out.max() <= 4096 and np.maximum(a.n_rev, a.n_fwd).max() <= 4096  # nothing cut off by the capacities
    for nm in ("status", "n_rev", "n_fwd", "n_out", "n_cart_out", "n_grid", "t_total", "t_rev", "s_last_sec",
               "out_sres", "theta_out", "cart_out", "hist", "flags", "row_offset"):
        x, y = getattr(a, nm), getattr(b, nm)
        assert (x is None) == (y is None), nm
        if x is not None:
            assert x.tobytes() == y.tobytes(), nm
    if ragged:
        for k in (0, B - 1):
            assert np.array_equal(a.rows(k), P.OracleRun(cfg, tres, th[k], None).theta), k
