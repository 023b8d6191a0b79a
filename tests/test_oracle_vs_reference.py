"""CPU: the oracle restatement against the UNMODIFIED reference sources, every stage bit for bit.

The reference's side of each comparison is oracle/_ref/libbatotp_ref.so where it is built
(`make -C oracle ref REF=<reference tree>`), and elsewhere the digests of its results stored in
tests/golden/reference_digests.json (_oracle.RefSide).  With the library built,
`BATOTP_RECORD_REF_DIGESTS=1 python -m pytest tests/test_oracle_vs_reference.py` rewrites that file."""
import ctypes as C

import numpy as np
import pytest

import _parity as P
from _oracle import Oracle, Ref, RefSide


@pytest.fixture
def ref(request):
    side = RefSide(request.node.name)
    yield side
    side.save()


def _cfg_bytes(cfg):
    return bytes(C.string_at(C.byref(cfg), C.sizeof(cfg)))


def _pair(ref, name, tmp_path, auto=False):
    d = P.GOLD + "/stock/" + name + "/"
    r = ref.call(lambda: Ref(d + "config.dat", d, str(tmp_path) + "/", auto_integ_res=auto))
    assert ref.same("load_file", lambda: r.load_file(), 0)
    cfg, tres, th, ca, ts = P.load_stock(name)
    if auto:
        cfg = cfg.copy()
        cfg.is_auto_integ_res = 1
    assert ref.same("cfg", lambda: _cfg_bytes(r.cfg()), _cfg_bytes(cfg)), \
        "Python config parser disagrees with BA::readConfigData"
    o = Oracle(cfg)
    n0 = (th if th is not None else ca).shape[2]
    o.load_raw(n0, tres, None if th is None else th[0], None if ca is None else ca[0], None if ts is None else ts[0])
    return cfg, r, o


def _sweeps(ref, r, o):
    for d, last in ((-1, 0), (1, 1)):
        assert o.sweep(d, last) == 0 and ref.same("sweep%d" % d, lambda: r.sweep(d, last), 0)
        assert ref.same("sMVC%d" % d, lambda: r.vec("sMVC"), o.vec("sMVC"))
        assert ref.same("sdot%d" % d, lambda: r.vec("sdot"), o.vec("sdot"))


@pytest.mark.parametrize("name", P.STOCK)
def test_every_stage_matches_bit_for_bit(ref, name, tmp_path):
    cfg, r, o = _pair(ref, name, tmp_path)
    J = cfg.n_joints
    assert o.interp_input() == 0 and ref.same("interp_input", lambda: r.interp_input(), 0)
    assert ref.same("nPts", lambda: r.scalar("nPts"), o.scalar("nPts"))
    for nm in ("theta", "thetaD", "thetaD2", "thetaC_y", "thetaC_m"):
        for j in range(J):
            # the last coefficient slot is never written (spline.cpp:203)
            cut = -1 if nm.startswith("thetaC") else None
            assert ref.same("in/%s/%d" % (nm, j), lambda: r.vec(nm, j)[:cut], o.vec(nm, j)[:cut]), (nm, j)
    if cfg.is_trq_on:
        for nm in ("a1", "a2", "a3", "a4", "a1C_m", "a4C_m"):
            for j in range(J):
                cut = -1 if nm.endswith("_m") else None
                assert ref.same("dyn/%s/%d" % (nm, j), lambda: r.vec(nm, j)[:cut], o.vec(nm, j)[:cut]), (nm, j)
    _sweeps(ref, r, o)
    assert ref.same("tTotalTraj", lambda: r.scalar("tTotalTraj"), o.scalar("tTotalTraj"))
    assert ref.same("sLastSec", lambda: r.scalar("sLastSec"), o.scalar("sLastSec"))
    ref.call(lambda: r.interp_output())
    o.interp_output()
    rows = {"theta": J}
    for nm, count in (("cart", "cartRows"), ("trq", "trqRows")):
        rows[nm] = int(o.scalar(count))
        assert ref.same(count, lambda: r.scalar(count), float(rows[nm]))
    for nm, n in rows.items():
        for j in range(n):
            assert ref.same("out/%s/%d" % (nm, j), lambda: r.vec(nm, j), o.vec(nm, j)), (nm, j)


@pytest.mark.parametrize("name", P.STOCK)
def test_switching_flags_match_instrumented_reference(ref, name, tmp_path):
    """The per-step switching flags: the reference's own per-point functions driven by the harness
    loop (ref_sweep_flags) must (a) reproduce BA::sweep's history bit for bit and (b) give the
    flags the oracle records."""
    cfg, r, o = _pair(ref, name, tmp_path)
    assert o.interp_input() == 0 and ref.same("interp_input", lambda: r.interp_input(), 0)
    got = ref.call(lambda: r.sweep_flags(-1))
    s, sd, fl = got if got else (None, None, None)
    assert o.sweep(-1, 0) == 0
    hs, hsd = o.vec("hist_s0"), o.vec("hist_sdot0")
    assert ref.same("rev/len", lambda: len(s), len(hs))
    # integration order vs ascending-s storage; the last integrated point is snapped afterwards
    assert ref.same("rev/s", lambda: s[:-1][::-1], hs[1:]) and ref.same("rev/sdot", lambda: sd[:-1][::-1], hsd[1:])
    assert ref.same("rev/flags", lambda: fl, o.vec("flags0").astype(np.uint8))
    # the real reverse sweep, to set up the forward pass identically
    assert ref.same("sweep-1", lambda: r.sweep(-1, 0), 0)
    got = ref.call(lambda: r.sweep_flags(1))
    s, sd, fl = got if got else (None, None, None)
    assert o.sweep(1, 1) == 0
    assert ref.same("fwd/s", lambda: s[:-1], o.vec("hist_s1")[:-1])
    assert ref.same("fwd/sdot", lambda: sd[:-1], o.vec("hist_sdot1")[:-1])
    assert ref.same("fwd/flags", lambda: fl, o.vec("flags1").astype(np.uint8))


@pytest.mark.parametrize("name", ["RR", "UR5", "KUKA-LWR-IV", "CSPR3DOF"])
def test_automatic_integration_resolution_matches(ref, name, tmp_path):
    """_isAutoIntegRes = true (the library default, ba.h:309; batest switches it off): adjust_s rewrites
    sWeights / scaleType / integRes per trajectory (ba.cpp:471-556).  The restatement must follow the unmodified
    reference through all three phases bit for bit.  (The generic robot has no Cartesian path to derive the
    resolution from: both sides reject GEN7DOF in this mode.)"""
    cfg, r, o = _pair(ref, name, tmp_path, auto=True)
    J = cfg.n_joints
    assert o.interp_input() == 0 and ref.same("interp_input", lambda: r.interp_input(), 0)
    assert ref.same("nPts", lambda: r.scalar("nPts"), o.scalar("nPts"))
    assert ref.same("integRes", lambda: r.scalar("integRes"), o.scalar("integRes"))
    _sweeps(ref, r, o)
    assert ref.same("tTotalTraj", lambda: r.scalar("tTotalTraj"), o.scalar("tTotalTraj"))
    ref.call(lambda: r.interp_output())
    o.interp_output()
    assert ref.same("outRes", lambda: r.scalar("outRes"), o.scalar("outRes"))
    for j in range(J):
        assert ref.same("out/theta/%d" % j, lambda: r.vec("theta", j), o.vec("theta", j)), j
    n_cart = int(o.scalar("cartRows"))
    assert ref.same("cartRows", lambda: r.scalar("cartRows"), float(n_cart))
    for j in range(n_cart):
        assert ref.same("out/cart/%d" % j, lambda: r.vec("cart", j), o.vec("cart", j)), j


def test_interpolation_only_mode_matches(ref, tmp_path):
    """_isInterpOnly (ba.cpp:139-159): interpInputData only re-samples the path at outRes and returns -1.  UR5 is
    the stock folder that carries both joint and Cartesian rows (the reference reads traj.cart[i] of an empty
    vector for the joint-only files in this mode, so those have no defined result)."""
    d = P.GOLD + "/stock/UR5/"
    r = ref.call(lambda: Ref(d + "config.dat", d, str(tmp_path) + "/"))
    ref.call(lambda: r.set_interp_only(True))
    assert ref.same("load_file", lambda: r.load_file(), 0)
    cfg, tres, th, ca, ts = P.load_stock("UR5")
    cfg = cfg.copy()
    cfg.is_interp_only = 1
    o = Oracle(cfg)
    o.load_raw(th.shape[2], tres, th[0], ca[0], None if ts is None else ts[0])
    assert o.interp_input() == -1 and ref.same("interp_input", lambda: r.interp_input(), -1)
    assert ref.same("nPts", lambda: r.scalar("nPts"), o.scalar("nPts"))
    assert o.scalar("sres") == cfg.out_res and ref.same("sres", lambda: r.scalar("sres"), o.scalar("sres"))
    for j in range(cfg.n_joints):
        assert ref.same("theta/%d" % j, lambda: r.vec("theta", j), o.vec("theta", j)), j
    assert int(o.scalar("cartRows")) == 6 and ref.same("cartRows", lambda: r.scalar("cartRows"), 6.0)
    for j in range(6):
        assert ref.same("cart/%d" % j, lambda: r.vec("cart", j), o.vec("cart", j)), j


def test_batch_runner_agrees(ref, tmp_path):
    from _oracle import orc_lib, ref_lib
    B = 12
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 500, B)
    cfgp = (P.GOLD + "/synthetic/GEN7DOF_config.dat").encode()
    fp, dp, ip = C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_int)

    def run(fn, first):
        tt = np.zeros(B); nr = np.zeros(B, np.int32); nf = np.zeros(B, np.int32); no = np.zeros(B, np.int32)
        st = np.zeros(B, np.int32); out = np.zeros((B, 7, 4096), np.float32)
        el = fn(first, B, th.shape[2], tres, th.ctypes.data_as(fp), None, 2, tt.ctypes.data_as(dp),
                nr.ctypes.data_as(ip), nf.ctypes.data_as(ip), no.ctypes.data_as(ip), st.ctypes.data_as(ip),
                out.ctypes.data_as(fp), 4096)
        assert el > 0
        return tt, nr, nf, no, st, out

    ref_out = ref.call(lambda: run(ref_lib().ref_batch_run, cfgp))
    orc_out = run(orc_lib().orc_batch_run, C.byref(cfg))
    for k, nm in enumerate(("t_total", "n_rev", "n_fwd", "n_out", "status", "rows")):
        assert ref.same(nm, lambda: ref_out[k], orc_out[k]), nm


@pytest.mark.parametrize("name", ["GEN7DOF", "RR", "UR5", "CSPR3DOF", "KUKA-LWR-IV"])
@pytest.mark.parametrize("decim,window", [(3, 1), (1, 3), (3, 3), (2, 4)])
def test_input_decimation_and_smoothing_match(ref, name, decim, window, tmp_path):
    """inputDecimFact > 1 / smoothWindow > 1 (ba.cpp:195-242 with util.cpp:254-288 smooth and 343-352 decimate;
    quirk Q6: the smoothWindow branch smooths with inputDecimFact as the window): no shipped config switches them
    on, so the restatement is pinned here against the unmodified reference, all three phases bit for bit."""
    d = P.GOLD + "/stock/" + name + "/"
    cfgp = P.variant_config(name, tmp_path, inputDecimFact=decim, smoothWindow=window)
    r = ref.call(lambda: Ref(cfgp, d, str(tmp_path) + "/"))
    assert ref.same("load_file", lambda: r.load_file(), 0)
    cfg, tres, th, ca, ts = P.load_stock_variant(name, tmp_path, inputDecimFact=decim, smoothWindow=window)
    assert ref.same("cfg", lambda: _cfg_bytes(r.cfg()), _cfg_bytes(cfg))
    assert cfg.input_decim_fact == decim and cfg.smooth_window == window
    o = Oracle(cfg)
    n0 = (th if th is not None else ca).shape[2]
    o.load_raw(n0, tres, None if th is None else th[0], None if ca is None else ca[0], None if ts is None else ts[0])
    J = cfg.n_joints
    oi = o.interp_input()
    assert ref.same("interp_input", lambda: r.interp_input(), oi)
    if oi != 0:
        return
    assert ref.same("nPts", lambda: r.scalar("nPts"), o.scalar("nPts"))
    for nm in ("theta", "thetaD", "thetaD2"):
        for j in range(J):
            assert ref.same("in/%s/%d" % (nm, j), lambda: r.vec(nm, j), o.vec(nm, j)), (nm, j)
    _sweeps(ref, r, o)
    assert ref.same("tTotalTraj", lambda: r.scalar("tTotalTraj"), o.scalar("tTotalTraj"))
    ref.call(lambda: r.interp_output())
    o.interp_output()
    for j in range(J):
        assert ref.same("out/theta/%d" % j, lambda: r.vec("theta", j), o.vec("theta", j)), j
    n_cart = int(o.scalar("cartRows"))
    assert ref.same("cartRows", lambda: r.scalar("cartRows"), float(n_cart))
    for j in range(n_cart):
        assert ref.same("out/cart/%d" % j, lambda: r.vec("cart", j), o.vec("cart", j)), j


@pytest.mark.parametrize("name", P.STOCK)
@pytest.mark.parametrize("start", [1.0e3, 0.5])
def test_per_sample_mvc_is_the_reference_functions(ref, name, start, tmp_path):
    """SURVEY 8a A10: the per-sample maximum-velocity curve has no reference output of its own; it is DEFINED as
    the reference's private per-point functions (evalSplinePartials, sdotLim, applyAccelConstraintsBisectionPt)
    evaluated at every knot.  ref_mvc_per_sample drives exactly those (oracle/ref_harness.cpp); the restatement
    must agree bit for bit on every robot: joint limits (GEN7DOF), Cartesian (UR5, KUKA), serial torque (RR),
    Par2Ser torque (CSPR3DOF)."""
    cfg, r, o = _pair(ref, name, tmp_path)
    assert o.interp_input() == 0 and ref.same("interp_input", lambda: r.interp_input(), 0)
    b = o.mvc_per_sample(start)
    assert len(b) == int(o.scalar("nPtsC")) and len(b) > 100
    assert ref.same("mvc", lambda: r.mvc_per_sample(start), b)
    assert np.isfinite(b).all() and b.max() <= start


def test_caller_supplied_dynamics_reproduce_the_reference_on_rr(ref, tmp_path):
    """cfg.dyn_source = 1: a1..a4 come from the caller's point function instead of Robot::call_dynSerial.  With
    dynRR restated behind that signature (orc_demo_dyn_rr) the plug-in path of the restatement must give what the
    unmodified reference gives with its built-in model: grid tables, both sweeps, torque rows - bit for bit."""
    from _oracle import dyn_fn_address
    cfg, r, o = _pair(ref, "RR", tmp_path)
    cfg2 = cfg.copy()
    cfg2.dyn_source = 1
    o = Oracle(cfg2)
    _, tres, th, ca, ts = P.load_stock("RR")
    o.load_raw(th.shape[2], tres, th[0], None, None)
    o.set_dyn_callback(dyn_fn_address("orc_demo_dyn_rr"))
    assert o.interp_input() == 0 and ref.same("interp_input", lambda: r.interp_input(), 0)
    for nm in ("a1", "a2", "a3", "a4", "a1C_m", "a4C_m"):
        for j in range(2):
            cut = -1 if nm.endswith("_m") else None
            assert ref.same("dyn/%s/%d" % (nm, j), lambda: r.vec(nm, j)[:cut], o.vec(nm, j)[:cut]), (nm, j)
    _sweeps(ref, r, o)
    ref.call(lambda: r.interp_output())
    o.interp_output()
    for nm in ("theta", "trq"):
        for j in range(2):
            assert ref.same("out/%s/%d" % (nm, j), lambda: r.vec(nm, j), o.vec(nm, j)), (nm, j)


def test_parallel_torque_without_par2ser_matches(ref, tmp_path):
    """isPar2Ser = 0 on the CSPR3DOF folder (ba.cpp:1463-1491; no shipped config uses it): restatement against the
    unmodified reference, every phase bit for bit."""
    d = P.GOLD + "/stock/CSPR3DOF/"
    cfgp = P.variant_config("CSPR3DOF", tmp_path, isPar2Ser=0)
    r = ref.call(lambda: Ref(cfgp, d, str(tmp_path) + "/"))
    assert ref.same("load_file", lambda: r.load_file(), 0)
    cfg, tres, th, ca, ts = P.load_stock_variant("CSPR3DOF", tmp_path, isPar2Ser=0)
    o = Oracle(cfg)
    o.load_raw(ca.shape[2], tres, None, ca[0], None)
    assert o.interp_input() == 0 and ref.same("interp_input", lambda: r.interp_input(), 0)
    _sweeps(ref, r, o)
    assert ref.same("tTotalTraj", lambda: r.scalar("tTotalTraj"), o.scalar("tTotalTraj"))
    ref.call(lambda: r.interp_output())
    o.interp_output()
    for nm in ("theta", "trq"):
        for j in range(3):
            assert ref.same("out/%s/%d" % (nm, j), lambda: r.vec(nm, j), o.vec(nm, j)), (nm, j)
