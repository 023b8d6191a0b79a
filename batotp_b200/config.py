"""Host-side option and file-format handling (Python mirror of the C++ facade).

Mirrors, for the tests and the benchmark harness, what the reference does on the
host before and after the accelerated path:

* ``read_config``      — ``BA::readConfigData``  (batotp/ba.cpp:1942-2087)
* ``read_traj_bin``    — ``BA::trajReadBIN``     (batotp/ba.cpp:2257-2312)
* ``read_traj_csv``    — ``BA::trajReadCSV``     (batotp/ba.cpp:2322-2461)
* ``pack_traj_out``    — ``BA::trajWriteBIN``    (batotp/ba.cpp:2582-2651)
* ``pack_s_sdot``      — ``BA::sdotWrite``       (batotp/ba.cpp:2726-2759)

``BatotpCfg`` is the ctypes image of ``struct batotp_cfg`` (include/batotp_cfg.h).
"""
from __future__ import annotations

import ctypes as C
import math
import struct
from typing import List, Optional, Tuple

import numpy as np

MAX_DOF = 7
KUKA, UR, RR, CSPR3DOF, GENJNT = 1, 2, 3, 4, 5
JOINT, CART, BOTH = 1, 2, 3
ROBOT_CODES = {"KUKA": KUKA, "UR": UR, "RR": RR, "CSPR3DOF": CSPR3DOF, "GENJNT": GENJNT}
PATH_CODES = {"JOINT": JOINT, "CART": CART, "BOTH": BOTH}


class BatotpCfg(C.Structure):
    _fields_ = [
        ("robot_type", C.c_int), ("is_parallel", C.c_int), ("n_joints", C.c_int), ("n_cart", C.c_int),
        ("is_bin_file", C.c_int), ("path_type", C.c_int), ("are_jnt_deg", C.c_int),
        ("is_jnt_vel_on", C.c_int), ("is_jnt_acc_on", C.c_int), ("is_trq_on", C.c_int),
        ("is_cart_vel_on", C.c_int), ("is_cart_acc_on", C.c_int), ("input_decim_fact", C.c_int),
        ("smooth_window", C.c_int), ("is_sdot_out", C.c_int), ("scale_type", C.c_int),
        ("is_svd", C.c_int), ("is_par2ser", C.c_int), ("is_interp_only", C.c_int),
        ("is_auto_integ_res", C.c_int), ("trig_mode", C.c_int), ("dyn_source", C.c_int), ("reserved_i", C.c_int * 10),
        ("jnt_vel_max", C.c_double * MAX_DOF), ("jnt_acc_max", C.c_double * MAX_DOF),
        ("jnt_trq_max", C.c_double * MAX_DOF), ("jnt_trq_min", C.c_double * MAX_DOF),
        ("cart_vel_max", C.c_double), ("cart_acc_max", C.c_double), ("integ_res", C.c_double),
        ("max_integ_time", C.c_double), ("jnt_thresh", C.c_double), ("cart_thresh", C.c_double),
        ("s_weights", C.c_double * 3), ("theta_norm_res", C.c_double), ("theta_norm_res2", C.c_double),
        ("cart_norm_res", C.c_double), ("cart_norm_res2", C.c_double), ("out_res", C.c_double),
        ("out_smooth_fact", C.c_double), ("reserved_d", C.c_double * 8),
    ]

    def copy(self) -> "BatotpCfg":
        c = BatotpCfg()
        C.memmove(C.byref(c), C.byref(self), C.sizeof(BatotpCfg))
        return c


# The limit members of batotp_cfg in the order of struct batotp_limits (include/batotp_cuda.h): one row of 30 doubles
LIMIT_FIELDS = (("jnt_vel_max", MAX_DOF), ("jnt_acc_max", MAX_DOF), ("jnt_trq_max", MAX_DOF), ("jnt_trq_min", MAX_DOF),
                ("cart_vel_max", 1), ("cart_acc_max", 1))
LIMIT_WIDTH = sum(n for _, n in LIMIT_FIELDS)


def limit_row(cfg: BatotpCfg) -> np.ndarray:
    """The limits of ``cfg`` as one float64 row of LIMIT_WIDTH values (batotp_limits order): scale it to build the
    per-trajectory rows of a batch (``Context.make_in(..., limits=)``)."""
    out = []
    for nm, n in LIMIT_FIELDS:
        v = getattr(cfg, nm)
        out += list(v) if n > 1 else [v]
    return np.array(out, dtype=np.float64)


def with_limits(cfg: BatotpCfg, row) -> BatotpCfg:
    """A copy of ``cfg`` whose limit members are replaced by ``row`` (LIMIT_WIDTH values, batotp_limits order), with
    the config reader's rule for a NaN jnt_trq_min: what a trajectory of a batch with that row is computed under."""
    row = np.asarray(row, dtype=np.float64).reshape(LIMIT_WIDTH)
    c = cfg.copy()
    k = 0
    for nm, n in LIMIT_FIELDS:
        if n > 1:
            arr = getattr(c, nm)
            for i in range(n):
                arr[i] = float(row[k + i])
        else:
            setattr(c, nm, float(row[k]))
        k += n
    for i in range(MAX_DOF):
        if math.isnan(c.jnt_trq_min[i]):
            c.jnt_trq_min[i] = -c.jnt_trq_max[i]
    return c


def _payload_lines(path: str) -> List[str]:
    with open(path, "r") as f:
        return f.read().split("\n")


def read_config(path: str) -> Tuple[BatotpCfg, str]:
    """Parse a ``config.dat``.  Returns (cfg, trajFileName).

    Follows the positional reader of ba.cpp:1958-2059: three header lines are skipped,
    then each option is the first whitespace-separated token(s) of its line, the rest
    of the line being a comment; two lines are skipped before each section.
    Raises ValueError where the reference returns -1.
    """
    lines = _payload_lines(path)
    pos = [3]

    def take() -> List[str]:
        ln = lines[pos[0]]
        pos[0] += 1
        return ln.split("//")[0].split()

    def skip(n: int) -> None:
        pos[0] += n

    cfg = BatotpCfg()
    robot = take()[0]
    if robot not in ROBOT_CODES:
        raise ValueError("robotType is %s" % robot)
    cfg.robot_type = ROBOT_CODES[robot]
    cfg.is_parallel = int(int(take()[0]) == 1)
    cfg.n_joints = int(take()[0])
    cfg.n_cart = int(take()[0])
    traj_name = take()[0]
    cfg.is_bin_file = int(int(take()[0]) == 1)
    ptype = take()[0]
    if ptype not in PATH_CODES:
        raise ValueError("pathType is %s" % ptype)
    cfg.path_type = PATH_CODES[ptype]
    skip(2)
    J = cfg.n_joints

    def flt(tok: str) -> float:
        return float("nan") if tok.upper().startswith("NAN") else float(tok)

    cfg.are_jnt_deg = int(int(take()[0]) == 1)
    cfg.is_jnt_vel_on = int(int(take()[0]) == 1)
    v = take()
    for i in range(J):
        cfg.jnt_vel_max[i] = flt(v[i])
    cfg.is_jnt_acc_on = int(int(take()[0]) == 1)
    v = take()
    for i in range(J):
        cfg.jnt_acc_max[i] = flt(v[i])
    cfg.is_trq_on = int(int(take()[0]) == 1)
    v = take()
    for i in range(J):
        cfg.jnt_trq_max[i] = flt(v[i])
    v = take()
    for i in range(J):
        x = flt(v[i])
        cfg.jnt_trq_min[i] = -cfg.jnt_trq_max[i] if math.isnan(x) else x  # ba.cpp:2020-2028
    cfg.is_cart_vel_on = int(int(take()[0]) == 1)
    cfg.cart_vel_max = flt(take()[0])
    cfg.is_cart_acc_on = int(int(take()[0]) == 1)
    cfg.cart_acc_max = flt(take()[0])
    skip(2)
    cfg.integ_res = flt(take()[0])
    cfg.max_integ_time = flt(take()[0])
    skip(2)
    cfg.input_decim_fact = int(take()[0])
    cfg.smooth_window = int(take()[0])
    cfg.is_sdot_out = int(int(take()[0]) == 1)
    cfg.jnt_thresh = flt(take()[0])
    cfg.cart_thresh = flt(take()[0])
    w = [flt(x) for x in take()[:3]]
    cfg.scale_type = int(take()[0])
    cfg.theta_norm_res = flt(take()[0])
    cfg.theta_norm_res2 = flt(take()[0])
    cfg.cart_norm_res = flt(take()[0])
    cfg.cart_norm_res2 = flt(take()[0])
    cfg.out_res = flt(take()[0])
    cfg.out_smooth_fact = flt(take()[0])
    cfg.is_svd = int(int(take()[0]) == 1)
    cfg.is_par2ser = int(int(take()[0]) == 1)
    wsum = w[0] + w[1] + w[2]  # ba.cpp:2063-2073
    if wsum <= 0:
        raise ValueError("sum(sWeights) should be greater than 0")
    for i in range(3):
        cfg.s_weights[i] = w[i] / wsum
    cfg.is_auto_integ_res = 0  # batest (test/main.cpp:53)
    cfg.is_interp_only = 0
    cfg.trig_mode = 1
    return cfg, traj_name


def read_traj_bin(path: str, n_joints: int, n_cart: int):
    """ba.cpp:2257-2312 -> (tres, n0, theta[J,n0] f32 or None, cart[C,n0] f32 or None)."""
    raw = open(path, "rb").read()
    tres = struct.unpack_from("<f", raw, 0)[0]
    n0 = struct.unpack_from("<i", raw, 4)[0]
    off = 8
    theta = cart = None
    is_theta = struct.unpack_from("<i", raw, off)[0]
    off += 4
    if is_theta == 1:
        theta = np.frombuffer(raw, dtype="<f4", count=n_joints * n0, offset=off).reshape(n_joints, n0).copy()
        off += 4 * n_joints * n0
    is_cart = struct.unpack_from("<i", raw, off)[0]
    off += 4
    if is_cart == 1:
        cart = np.frombuffer(raw, dtype="<f4", count=n_cart * n0, offset=off).reshape(n_cart, n0).copy()
        off += 4 * n_cart * n0
    return float(tres), int(n0), theta, cart


def read_traj_csv(path: str, n_joints: int, n_cart: int, is_generic: bool):
    """ba.cpp:2322-2461 -> (tres, n0, theta f64 or None, cart f64 or None, timestamp f64, header)."""
    with open(path, "r") as f:
        lines = [ln for ln in f.read().split("\n")]
    header = [h.strip() for h in lines[0].replace("\t", " ").split(",") if h.strip()]
    rows = []
    for ln in lines[1:]:
        toks = [x for x in ln.replace(",", " ").split()]
        if not toks:
            break
        try:
            rows.append([float(x) for x in toks])
        except ValueError:
            break
    n0 = len(rows)
    nf = n_joints if is_generic else n_joints + n_cart + 1
    header = header[:nf]
    is_ts = "timestamp" in header
    is_j = "j1" in header
    is_c = "x" in header
    a = np.array(rows, dtype=np.float64)
    col = 0
    ts = None
    theta = cart = None
    if is_ts:
        ts = a[:, col].copy()
        col += 1
    if is_j:
        theta = np.ascontiguousarray(a[:, col:col + n_joints].T)
        col += n_joints
    if is_c:
        cart = np.ascontiguousarray(a[:, col:col + n_cart].T)
        col += n_cart
    if ts is None:
        ts = 0.2 * np.arange(n0, dtype=np.float64)  # ba.cpp:2440-2444
    tres = ts[-1] / (n0 - 1)
    return float(tres), n0, theta, cart, ts, header


def pack_traj_out(sres: float, n_pts: int, theta, cart=None, trq=None) -> bytes:
    """ba.cpp:2617-2647: f32 sres; u32 nPts; i32 1; J rows f32; i32 isCart; [C rows]; i32 isTrq; [J rows]."""
    out = [struct.pack("<f", np.float32(sres)), struct.pack("<I", n_pts), struct.pack("<i", 1)]
    out.append(np.asarray(theta, dtype=np.float64).astype("<f4").tobytes())
    out.append(struct.pack("<i", 1 if cart is not None else 0))
    if cart is not None:
        out.append(np.asarray(cart, dtype=np.float64).astype("<f4").tobytes())
    out.append(struct.pack("<i", 1 if trq is not None else 0))
    if trq is not None:
        out.append(np.asarray(trq, dtype=np.float64).astype("<f4").tobytes())
    return b"".join(out)


def pack_s_sdot(sres: float, hists) -> bytes:
    """ba.cpp:2735-2749: for rev then fwd: f64 sres; i32 n; n f32 s; n f32 sdot."""
    out = []
    for s, sd in hists:
        out.append(struct.pack("<d", sres))
        out.append(struct.pack("<i", len(s)))
        out.append(np.asarray(s, dtype=np.float64).astype("<f4").tobytes())
        out.append(np.asarray(sd, dtype=np.float64).astype("<f4").tobytes())
    return b"".join(out)
