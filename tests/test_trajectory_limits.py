"""Per-trajectory limits (batotp_batch_in.limits): trajectory b of a batch with limit rows must give exactly what a
run of its own gives under the batch cfg with b's limits.  The CPU half runs the host-emulation build of the kernels
(the k_sweep / k_sweep_group / k_mvc instantiations that read the rows), the `-m gpu` half the product library on the
device, where the machine-filling sizes are checked too."""
import ctypes as C

import numpy as np
import pytest

import _parity as P
from batotp_b200 import native
from batotp_b200.config import LIMIT_WIDTH, limit_row, with_limits

ST_UNSUPPORTED = 512
ARRAYS = ("status", "n_rev", "n_fwd", "n_out", "n_cart_out", "n_grid", "t_total", "t_rev", "s_last_sec", "out_sres",
          "theta_out", "cart_out", "trq_out", "hist", "flags")
# the regimes of test_limit_regimes_match_oracle (acceleration, velocity scaling)
REGIMES = [(0.05, 1.0), (20.0, 0.2), (1.0, 5.0), (1.0, 1.0), (300.0, 30.0)]
J0, A0, T0, M0, CV, CA = 0, 7, 14, 21, 28, 29  # offsets of the members in a limit row


@pytest.fixture(scope="module")
def emu():
    import __graft_entry__ as g
    c = native.Context(0, g.build_emu())
    c.set_sweep_kernel(1)  # the group kernel's shuffles are slow under the emulation: asked for where it is tested
    yield c
    c.close()


@pytest.fixture(scope="module")
def gpu():
    c = native.Context(0)  # product library; raises without a CUDA device
    yield c
    c.close()


@pytest.fixture(params=["emu", pytest.param("gpu", marks=pytest.mark.gpu)])
def ctx(request):
    return request.getfixturevalue(request.param)


@pytest.fixture(params=[1, 2], ids=["lane_kernel", "group_kernel"])
def sweep_kernel(request, ctx):
    """Both sweep kernels: 1 = one trajectory per lane (k_sweep.cuh), 2 = a group of lanes per trajectory
    (k_sweep_group.cuh).  The emulation context is left on the lane kernel afterwards, the device one on automatic."""
    ctx.set_sweep_kernel(request.param)
    yield request.param
    ctx.set_sweep_kernel(1 if ctx.L._name.endswith("libbatotp_emu.so") else 0)


@pytest.fixture(params=[1, 2], ids=["lane_kernel", "group_kernel"])
def gpu_sweep_kernel(request, gpu):
    """sweep_kernel for the tests that run on the device only."""
    gpu.set_sweep_kernel(request.param)
    yield request.param
    gpu.set_sweep_kernel(0)


def mixed_rows(cfg, B, seed, regimes=REGIMES, joint_spread=(0.6, 1.6), cart=(1.0, 1.0), trq=(1.0, 1.0)):
    """One row per trajectory: a regime of test_limit_regimes_match_oracle in turn, times per-joint factors."""
    rng = np.random.RandomState(seed)
    base = limit_row(cfg)
    rows = np.tile(base, (B, 1))
    for b in range(B):
        acc, vel = regimes[b % len(regimes)]
        rows[b, A0:A0 + 7] *= acc * rng.uniform(*joint_spread, 7)
        rows[b, J0:J0 + 7] *= vel * rng.uniform(*joint_spread, 7)
        f = rng.uniform(*trq, 7)
        rows[b, T0:T0 + 7] *= f
        rows[b, M0:M0 + 7] *= f
        rows[b, CV] *= rng.uniform(*cart)
        rows[b, CA] *= rng.uniform(*cart)
    return rows


def run(ctx, cfg, tres, th, ca, ts=None, limits=None, n0=None, out_cap=32768, hist_cap=32768):
    ref = th if th is not None else ca
    bi = ctx.make_in(th, ca, tres, n0=n0, timestamp=ts, limits=limits)
    res = native.BatchResult(ref.shape[0], cfg.n_joints, cfg.n_cart, out_cap, hist_cap, bool(cfg.is_trq_on))
    ctx.optimize_batch(cfg, bi, res)
    return res


def same(a, b, idx=None):
    for nm in ARRAYS:
        x, y = getattr(a, nm), getattr(b, nm)
        if x is None:
            assert y is None, nm
            continue
        if idx is not None:
            x, y = x[idx], y
        assert np.array_equal(x, y), nm


def check_oracle(cfg, res, rows, tres, th, ca, idx, ts=None, dyn_fn=None):
    for b in idx:
        c = with_limits(cfg, rows[b])
        orc = P.OracleRun(c, tres, None if th is None else th[b], None if ca is None else ca[b],
                          None if ts is None else ts[0], dyn_fn=dyn_fn)
        assert orc.ok, b
        assert res.status[b] & native.ST_FATAL_MASK == 0, (b, res.status[b])
        assert P.compare(c, res, b, orc) == [], b


def tile1(a, B):
    return None if a is None else np.ascontiguousarray(np.repeat(a, B, axis=0))


# ----------------------------------------------------------------------------- 1. rows equal to the cfg
@pytest.mark.parametrize("name", P.STOCK + ["synthetic GEN7DOF"])
def test_rows_equal_to_the_cfg_change_nothing(ctx, name):
    if name in P.STOCK:
        cfg, tres, th, ca, ts = P.load_stock(name)
    else:
        cfg, tres, th, ca = P.load_synth("GEN7DOF", 200, 6)
        ts = None
    B = (th if th is not None else ca).shape[0]
    rows = np.tile(limit_row(cfg), (B, 1))
    ctx.stats_reset()
    a = run(ctx, cfg, tres, th, ca, ts)
    sa = ctx.stats()
    ctx.stats_reset()
    b = run(ctx, cfg, tres, th, ca, ts, limits=rows)
    sb = ctx.stats()
    same(a, b)
    for k in ("verifies", "steps", "trajectories"):
        assert sa[k] == sb[k], k


# ----------------------------------------------------------------------------- 2. the filtered kernel, mixed regimes
def test_mixed_regimes_match_oracle_with_clean_certificates(emu):
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 900, 10)
    rows = mixed_rows(cfg, 10, 1)
    st = (C.c_longlong * 16)()
    emu.L.batotp_emu_filter_stats(st, 16, 1)
    res = run(emu, cfg, tres, th, None, limits=rows, out_cap=65536, hist_cap=65536)
    emu.L.batotp_emu_filter_stats(st, 16, 1)
    check_oracle(cfg, res, rows, tres, th, None, range(10))
    certain, exact, b_joint, b_exact, v_skip, v_one, v_all = list(st)[:7]
    # every shortcut agreed with the full exact computation on the trajectory's own row (TEST-ONLY blocks)
    assert list(st)[8:11] == [0, 0, 0], list(st)
    assert certain > 100000
    assert exact < 0.01 * certain
    assert b_exact < 0.001 * b_joint
    assert v_all < 0.001 * (v_skip + v_one + 1)


def test_mixed_regimes_both_kernels(ctx, sweep_kernel):
    B = 5 if ctx.L._name.endswith("libbatotp_emu.so") else 40
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 20000, B)
    rows = mixed_rows(cfg, B, 2)
    res = run(ctx, cfg, tres, th, None, limits=rows, out_cap=65536, hist_cap=65536)
    check_oracle(cfg, res, rows, tres, th, None, range(0, B, max(1, B // 10)))


# ----------------------------------------------------------------------------- 3. the other kernel configurations
def test_kuka_cartesian_limits(ctx):
    cfg, tres, th, _ = P.load_synth("KUKA", 10, 2)
    rows = mixed_rows(cfg, 2, 3, regimes=[(1.0, 1.0), (0.5, 1.5)], cart=(0.5, 1.5))
    res = run(ctx, cfg, tres, th, None, limits=rows, out_cap=49152, hist_cap=49152)
    check_oracle(cfg, res, rows, tres, th, None, range(2))


def test_rr_torque_limits(ctx, sweep_kernel):
    cfg, tres, th, ca, ts = P.load_stock("RR")
    B = 4
    rows = mixed_rows(cfg, B, 4, regimes=[(1.0, 1.0), (1.0, 0.7)], trq=(0.5, 1.3), cart=(0.6, 1.4))
    res = run(ctx, cfg, tres, tile1(th, B), tile1(ca, B), tile1(ts, B), limits=rows)
    check_oracle(cfg, res, rows, tres, tile1(th, B), tile1(ca, B), range(B), ts=ts)
    assert len(set(res.t_total.tolist())) == B  # the rows bind


@pytest.mark.parametrize("par2ser", [1, 0])
def test_cspr_torque_limits(ctx, par2ser, tmp_path):
    cfg, tres, th, ca, ts = P.load_stock_variant("CSPR3DOF", tmp_path, isPar2Ser=par2ser)
    B = 3
    rows = mixed_rows(cfg, B, 5, regimes=[(1.0, 1.0), (0.8, 0.9), (1.2, 1.1)], trq=(0.8, 1.2), cart=(0.7, 1.3))
    res = run(ctx, cfg, tres, tile1(th, B), tile1(ca, B), tile1(ts, B), limits=rows)
    check_oracle(cfg, res, rows, tres, tile1(th, B), tile1(ca, B), range(B))


def test_kuka_torque_variant_on_a_caller_model(ctx):
    from _oracle import dyn_fn_address
    cfg, tres, th, ca, ts = P.load_stock("KUKA-LWR-IV")
    c2 = cfg.copy()
    c2.is_trq_on = 1
    c2.dyn_source = 1
    for j, v in enumerate((60.0, 60.0, 30.0, 30.0, 15.0, 15.0, 8.0)):
        c2.jnt_trq_max[j] = v
        c2.jnt_trq_min[j] = -v
    B = 3
    rows = mixed_rows(c2, B, 6, regimes=[(1.0, 1.0)], trq=(0.6, 1.2), cart=(0.8, 1.2))
    fn = dyn_fn_address("orc_demo_dyn_serial")
    try:
        ctx.set_dyn_callback(fn)
        res = run(ctx, c2, tres, tile1(th, B), None, limits=rows)
    finally:
        ctx.set_dyn_callback(None)
    check_oracle(c2, res, rows, tres, tile1(th, B), None, range(B), dyn_fn=fn)


def test_ur5_automatic_step_follows_the_rows(ctx):
    cfg, tres, th, ca, ts = P.load_stock("UR5")
    cfg = cfg.copy()
    cfg.is_auto_integ_res = 1
    B = 3
    rows = mixed_rows(cfg, B, 7, regimes=[(1.0, 1.0), (3.0, 1.0), (0.3, 0.8)], cart=(0.7, 1.5))
    res = run(ctx, cfg, tres, tile1(th, B), tile1(ca, B), tile1(ts, B), limits=rows)
    check_oracle(cfg, res, rows, tres, tile1(th, B), tile1(ca, B), range(B), ts=ts)


# ----------------------------------------------------------------------------- 4. re-slicing
def test_rows_survive_chunks_stragglers_and_the_tail_helper(ctx):
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 60, 11)
    rows = mixed_rows(cfg, 11, 8)
    ctx.set_tail_overlap(False)
    ctx.set_chunk(16384)
    try:
        ref = run(ctx, cfg, tres, th, None, limits=rows, out_cap=65536, hist_cap=65536)
        steps = np.maximum(ref.n_rev, ref.n_fwd)
        variants = []
        ctx.set_chunk(4)  # 4 + 4 + 3: the last chunk on the second context
        ctx.set_tail_overlap(True)
        variants.append(run(ctx, cfg, tres, th, None, limits=rows, out_cap=65536, hist_cap=65536))
        ctx.set_out_chunk(3)
        variants.append(run(ctx, cfg, tres, th, None, limits=rows, out_cap=65536, hist_cap=65536))
        ctx.set_step_hint(int(np.sort(steps)[-3]) - 1)  # stragglers on both contexts
        variants.append(run(ctx, cfg, tres, th, None, limits=rows, out_cap=65536, hist_cap=65536))
    finally:
        ctx.set_step_hint(0)
        ctx.set_out_chunk(8192)
        ctx.set_chunk(16384)
        ctx.set_tail_overlap(True)
    for v in variants:
        same(ref, v)
    perm = np.random.RandomState(9).permutation(11)
    p = run(ctx, cfg, tres, np.ascontiguousarray(th[perm]), None, limits=rows[perm], out_cap=65536, hist_cap=65536)
    for nm in ARRAYS:
        x = getattr(ref, nm)
        if x is not None:
            assert np.array_equal(x[perm], getattr(p, nm)), nm
    check_oracle(cfg, ref, rows, tres, th, None, (0, 4, 10))


def test_structured_rows_are_the_same_as_flat_rows(ctx):
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 70, 3)
    rows = mixed_rows(cfg, 3, 10)
    st = np.zeros(3, native.LIMITS_DTYPE)
    for nm, off, n in (("jnt_vel_max", J0, 7), ("jnt_acc_max", A0, 7), ("jnt_trq_max", T0, 7),
                       ("jnt_trq_min", M0, 7)):
        st[nm] = rows[:, off:off + n]
    st["cart_vel_max"], st["cart_acc_max"] = rows[:, CV], rows[:, CA]
    same(run(ctx, cfg, tres, th, None, limits=rows), run(ctx, cfg, tres, th, None, limits=st))
    with pytest.raises(ValueError):
        ctx.make_in(th, None, tres, limits=rows[:2])


# ----------------------------------------------------------------------------- 5. the row rules
def test_nan_torque_minimum_and_rejected_rows(ctx):
    cfg, tres, th, ca, ts = P.load_stock("RR")
    B = 6
    rows = mixed_rows(cfg, B, 11, regimes=[(1.0, 1.0)], trq=(0.7, 1.3))
    rows[:, M0:M0 + 7] = -rows[:, T0:T0 + 7]
    nanrows = rows.copy()
    nanrows[:, M0:M0 + 2] = np.nan  # the config reader's NaN: -JntTrqMax
    nanrows[:, J0 + 2:J0 + 7] = np.nan  # past nJoints: ignored
    nanrows[:, T0 + 2:T0 + 7] = np.inf
    nanrows[:, A0:A0 + 2] = -1.0    # jnt_acc_max is not used (acceleration limits off)
    args = (cfg, tres, tile1(th, B), tile1(ca, B), tile1(ts, B))
    good = run(ctx, *args, limits=rows)
    same(good, run(ctx, *args, limits=nanrows))
    bad = rows.copy()
    bad[1, J0 + 1] = 0.0        # a velocity maximum <= 0
    bad[3, T0] = np.inf         # a torque limit that is on and not finite
    bad[4, CV] = np.nan         # Cartesian velocity limit on
    r = run(ctx, *args, limits=bad)
    for b in range(B):
        if b in (1, 3, 4):
            assert r.status[b] == ST_UNSUPPORTED and r.n_out[b] == 0 and r.n_fwd[b] == 0, b
        else:
            for nm in ARRAYS:
                x = getattr(good, nm)
                if x is not None:
                    assert np.array_equal(x[b], getattr(r, nm)[b]), (nm, b)


# ----------------------------------------------------------------------------- 6. the per-sample MVC
@pytest.mark.parametrize("name", ["GEN7DOF", "RR", "CSPR3DOF"])
def test_per_sample_mvc_with_rows(ctx, name):
    from _oracle import Oracle
    cfg, tres, th, ca, ts = P.load_stock(name)
    B = 3
    rows = mixed_rows(cfg, B, 12, regimes=[(1.0, 1.0), (0.5, 0.7), (2.0, 1.5)], trq=(0.7, 1.3), cart=(0.7, 1.3))
    ctx.load(cfg, ctx.make_in(tile1(th, B), tile1(ca, B), tres, timestamp=tile1(ts, B), limits=rows))
    ctx.interp_input()
    n0 = (th if th is not None else ca).shape[2]
    for start in (1.0e3, 0.5):
        wants = []
        for b in range(B):
            o = Oracle(with_limits(cfg, rows[b]))
            o.load_raw(n0, tres, None if th is None else th[0], None if ca is None else ca[0],
                       None if ts is None else ts[0])
            assert o.interp_input() == 0
            wants.append(o.mvc_per_sample(start))
        got = ctx.mvc_per_sample(B, max(len(w) for w in wants) + 8, start)
        for b in range(B):
            assert np.array_equal(got[b, :len(wants[b])], wants[b]), (b, start)
        if start > 1.0:
            assert not np.array_equal(wants[0], wants[1])  # the rows bind


# ----------------------------------------------------------------------------- GPU: sizes that fill the machine
def _by_class(cfg, rows, classes, fn):
    for k in np.unique(classes):
        idx = np.nonzero(classes == k)[0]
        fn(with_limits(cfg, rows[idx[0]]), idx)


def _speed_classes(cfg, B, n_classes, seed, fmin):
    """A speed-override factor per path, drawn from n_classes values in [fmin, 1]: velocity x f, acceleration x f^2."""
    rng = np.random.RandomState(seed)
    f = np.linspace(fmin, 1.0, n_classes)
    cls = rng.randint(0, n_classes, B)
    rows = np.tile(limit_row(cfg), (B, 1))
    rows[:, J0:J0 + 7] *= f[cls, None]
    rows[:, A0:A0 + 7] *= (f[cls] ** 2)[:, None]
    rows[:, CV] *= f[cls]
    rows[:, CA] *= f[cls] ** 2
    return rows, cls


@pytest.mark.gpu
@pytest.mark.parametrize("name,B,fmin", [("GEN7DOF", 4096, 0.4), ("KUKA", 256, 0.7), ("CSPR3DOF", 1024, 0.4)])
def test_filled_machine_matches_oracle_per_limit_class(gpu, name, B, fmin, gpu_sweep_kernel):
    """(KUKA paths take ~18 600 steps per sweep at the stock limits: slower classes would reach the default step
    ceiling, which ends a trajectory where the reference would go on)"""
    from test_gpu_parity import _oracle_batch
    cfg, tres, th, ca = P.load_synth(name, 3000, B)
    rows, cls = _speed_classes(cfg, B, 8, 13, fmin)
    scal = native.BatchResult(B, cfg.n_joints, cfg.n_cart, 0, 0, bool(cfg.is_trq_on), want_rows=False, want_hist=False)
    gpu.optimize_batch(cfg, gpu.make_in(th, ca, tres, limits=rows), scal)
    assert (scal.status & native.ST_FATAL_MASK == 0).all()
    out_cap = int(scal.n_out.max()) + 8
    res = native.BatchResult(B, cfg.n_joints, cfg.n_cart, out_cap, 0, bool(cfg.is_trq_on), want_rows=True,
                             want_hist=False)
    gpu.optimize_batch(cfg, gpu.make_in(th, ca, tres, limits=rows), res)

    def check(c, idx):
        sub = lambda a: None if a is None else np.ascontiguousarray(a[idx])
        tt, nr, nf, no, st, rr = _oracle_batch(c, tres, sub(th), sub(ca), out_cap)
        assert (st == 0).all()
        assert np.array_equal(res.n_rev[idx], nr) and np.array_equal(res.n_fwd[idx], nf)
        assert np.array_equal(res.n_out[idx], no) and np.array_equal(res.t_total[idx], tt)
        assert np.array_equal(res.theta_out[idx], rr)

    _by_class(cfg, rows, cls, check)
    assert len(np.unique(res.t_total[cls == 0])) > 1 and res.t_total[cls == 0].mean() > res.t_total[cls == 7].mean()


@pytest.mark.gpu
def test_device_resident_inputs_and_results_and_ragged_rows_with_limits(gpu):
    import torch
    B, cap = 300, 32768
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 7000, B)
    rows = mixed_rows(cfg, B, 14)
    a = run(gpu, cfg, tres, th, None, limits=rows, out_cap=cap, hist_cap=cap)
    # payload in HBM, rows on the host
    dth = torch.from_numpy(th).cuda()
    bi = gpu.make_in(device_ptrs=dict(theta=dth.data_ptr(), B=B, n0_max=th.shape[2]), tres=tres, limits=rows)
    b = native.BatchResult(B, cfg.n_joints, cfg.n_cart, cap, cap, False)
    gpu.set_chunk(128)
    try:
        gpu.optimize_batch(cfg, bi, b)
    finally:
        gpu.set_chunk(0)
    same(a, b)
    # results into HBM
    dev = {}
    d = native.BatchResult(B, cfg.n_joints, cfg.n_cart, cap, cap, False)
    for nm in ("status", "n_rev", "n_fwd", "n_out", "t_total", "theta_out", "hist", "flags"):
        host = getattr(d, nm)
        dev[nm] = torch.zeros(host.shape, dtype=getattr(torch, str(host.dtype)), device="cuda:0")
        ptr = dev[nm].data_ptr()
        setattr(d.c, nm, ptr if nm in ("theta_out", "hist", "flags") else C.cast(ptr, type(getattr(d.c, nm))))
    for nm in ("n_cart_out", "n_grid", "t_rev", "s_last_sec", "out_sres", "cart_out"):
        setattr(d.c, nm, None)
    d.c.on_device = 1
    gpu.optimize_batch(cfg, gpu.make_in(th, None, tres, limits=rows), d)
    torch.cuda.synchronize()
    for nm, t in dev.items():
        assert np.array_equal(getattr(a, nm), t.cpu().numpy()), nm
    # ragged rows
    total = int(a.n_out.sum())
    r = native.BatchResult(B, cfg.n_joints, cfg.n_cart, 0, 0, False, want_hist=False, ragged_cap=total)
    gpu.optimize_batch(cfg, gpu.make_in(th, None, tres, limits=rows), r)
    for k in range(B):
        assert np.array_equal(r.rows(k), a.theta_out[k, :, :a.n_out[k]]), k
    check_oracle(cfg, a, rows, tres, th, None, range(0, B, 37))
