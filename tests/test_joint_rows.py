"""CPU (host emulation of the kernels): a joint-only generic robot stores only its joint rows.

Its Cartesian rows are zero throughout the reference's path, so the kernels read them as a literal 0.0 and the
packing writes +0.0 for them without a source row.  These tests pin what that must not change: the Cartesian
output bytes (+0.0, also in the FP64 side output), the arc-length arithmetic that still adds the zero Cartesian
norm (a non-zero Cartesian weight under each scale type), and the configurations that keep their Cartesian rows."""
import numpy as np
import pytest

import _parity as P
from batotp_b200 import native
from batotp_b200.config import BOTH


@pytest.fixture(scope="module")
def ctx():
    import __graft_entry__ as g
    c = native.Context(0, g.build_emu())
    c.set_sweep_kernel(1)  # the lane kernel: the group kernel's shuffles are slow under the emulation
    yield c
    c.close()


def _all_positive_zero(a):
    a = np.ascontiguousarray(a)
    return not a.view(np.uint32 if a.dtype == np.float32 else np.uint64).any()


@pytest.mark.parametrize("keep_f64", [False, True])
def test_gen7dof_cartesian_rows_are_positive_zero(ctx, keep_f64):
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 0, 3)
    assert cfg.n_cart == 3
    ctx.set_keep_f64(keep_f64)
    try:
        res = P.run_device(ctx, cfg, tres, th, None, out_cap=4096, hist_cap=4096)
        for b in range(3):
            orc = P.OracleRun(cfg, tres, th[b], None)
            assert P.compare(cfg, res, b, orc) == [], b
            assert res.status[b] & native.ST_FATAL_MASK == 0
            assert res.n_cart_out[b] > 0
            assert _all_positive_zero(res.cart_out[b]), b
            if keep_f64:
                n = int(res.n_out[b])
                for r in range(cfg.n_joints):
                    v = ctx.get_f64("theta_out", b, r)
                    assert len(v) == n and np.array_equal(v.astype(np.float32), orc.theta[r]), (b, r)
                for r in range(3):
                    v = ctx.get_f64("cart_out", b, r)
                    assert len(v) == res.n_cart_out[b] and _all_positive_zero(v), (b, r)
                    for nm in ("cartC_y", "cartC_m"):
                        v = ctx.get_f64(nm, b, r)
                        assert len(v) == res.n_grid[b] and _all_positive_zero(v), (nm, b, r)
    finally:
        ctx.set_keep_f64(False)


@pytest.mark.parametrize("scale_type", [0, 1, 2])
def test_joint_only_with_cartesian_weight_matches_oracle(ctx, scale_type):
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 5, 3)
    cfg = cfg.copy()
    cfg.scale_type = scale_type
    for i, v in enumerate((0.2, 0.5, 0.3)):  # time, joint and Cartesian weights
        cfg.s_weights[i] = v
    res = P.run_device(ctx, cfg, tres, th, None, out_cap=4096, hist_cap=4096)
    for b in range(3):
        orc = P.OracleRun(cfg, tres, th[b], None)
        assert P.compare(cfg, res, b, orc) == [], (b, res.status[b])


def test_generic_both_path_keeps_cartesian_rows(ctx):
    cfg, tres, th, _ = P.load_synth("GEN7DOF", 9, 2)
    cfg = cfg.copy()
    cfg.path_type = BOTH
    # Cartesian rows driven by the path: smooth functions of the joint rows
    ca = np.ascontiguousarray(np.stack([0.3 * np.sin(th[:, 0]), 0.2 * np.cos(th[:, 1]), 0.1 * th[:, 2]], axis=1))
    res = P.run_device(ctx, cfg, tres, th, ca, out_cap=4096, hist_cap=4096)
    for b in range(2):
        orc = P.OracleRun(cfg, tres, th[b], ca[b])
        assert orc.cart is not None and np.abs(orc.cart).max() > 0
        assert P.compare(cfg, res, b, orc) == [], (b, res.status[b])
        assert np.abs(res.cart_out[b, :, :res.n_cart_out[b]]).max() > 0
