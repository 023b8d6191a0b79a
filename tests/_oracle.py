"""ctypes access to the two test oracles (TEST INFRASTRUCTURE ONLY).

* ``Oracle``  — oracle/_build/libba_oracle.so, the C restatement (always buildable).
* ``Ref``     — oracle/_ref/libbatotp_ref.so, the unmodified reference sources compiled
                in place with the Eigen stand-in (``make -C oracle ref REF=<reference tree>``).
* ``RefSide`` — the reference's side of a comparison: ``Ref`` where it is built, the digests
                of its results stored in tests/golden/reference_digests.json elsewhere.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from batotp_b200.config import BatotpCfg  # noqa: E402

ORC_SO = os.path.join(ROOT, "oracle", "_build", "libba_oracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libbatotp_ref.so")
REF_DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_digests.json")

_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_ip = C.POINTER(C.c_int)


def build_oracles() -> None:
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "all"], check=True,
                   stdout=subprocess.DEVNULL)


def _ptr(a, typ):
    return None if a is None else a.ctypes.data_as(typ)


_orc = None


def orc_lib():
    global _orc
    if _orc is None:
        if not os.path.exists(ORC_SO):
            build_oracles()
        L = C.CDLL(ORC_SO)
        L.orc_new.restype = C.c_void_p
        L.orc_new.argtypes = [C.POINTER(BatotpCfg)]
        L.orc_free.argtypes = [C.c_void_p]
        L.orc_load_raw.argtypes = [C.c_void_p, C.c_int, C.c_double, _fp, _fp, _dp]
        L.orc_load_raw_f64.argtypes = [C.c_void_p, C.c_int, C.c_double, _dp, _dp, _dp]
        for f in ("orc_interp_input", "orc_interp_output", "orc_optimize"):
            getattr(L, f).argtypes = [C.c_void_p]
        L.orc_sweep.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.orc_mvc_per_sample.argtypes = [C.c_void_p, C.c_double, _dp, C.c_int]
        L.orc_set_dyn_callback.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_get_vec.argtypes = [C.c_void_p, C.c_char_p, C.c_int, _dp, C.c_int]
        L.orc_get_scalar.argtypes = [C.c_void_p, C.c_char_p]
        L.orc_get_scalar.restype = C.c_double
        L.orc_pack_traj_out.argtypes = [C.c_void_p, C.c_char_p, C.c_long]
        L.orc_pack_traj_out.restype = C.c_long
        L.orc_pack_s_sdot.argtypes = [C.c_void_p, C.c_char_p, C.c_long]
        L.orc_pack_s_sdot.restype = C.c_long
        L.orc_batch_run.restype = C.c_double
        L.orc_batch_run.argtypes = [C.POINTER(BatotpCfg), C.c_int, C.c_int, C.c_double, _fp, _fp, C.c_int,
                                    _dp, _ip, _ip, _ip, _ip, _fp, C.c_int]
        _orc = L
    return _orc


def dyn_fn_address(name: str) -> int:
    """Address of one of the oracle library's demonstration dynamics (orc_demo_dyn_rr, orc_demo_dyn_serial): the
    same host function feeds the oracle and - through batotp_cuda_set_dyn_callback - the device path."""
    return C.cast(getattr(orc_lib(), name), C.c_void_p).value


_ref = None


def ref_available() -> bool:
    return os.path.exists(REF_SO)


def digest(value) -> str:
    """dtype, shape and sha256[:16] of a result's bytes (Python numbers as float64, bytes as uint8)."""
    if isinstance(value, bytes):
        a = np.frombuffer(value, np.uint8)
    elif isinstance(value, np.ndarray):
        a = np.ascontiguousarray(value)
    else:
        a = np.asarray(value, dtype=np.float64)
    return "%s%s:%s" % (a.dtype.str, list(a.shape), hashlib.sha256(a.tobytes()).hexdigest()[:16])


class RefSide:
    """The reference's side of one test case's comparisons.

    Where oracle/_ref is built the reference library itself runs: ``same`` compares its result with the value and
    checks it against the stored digest (with BATOTP_RECORD_REF_DIGESTS=1 it stores the digest instead; ``save``
    writes the file).  Elsewhere the reference is not called at all and ``same`` compares the value's digest with
    the stored one, so the comparisons hold on every checkout."""

    def __init__(self, case: str):
        self.case = case
        self.live = ref_available()
        self.record = self.live and os.environ.get("BATOTP_RECORD_REF_DIGESTS") == "1"
        self.stored = json.load(open(REF_DIGESTS)).get(case, {}) if os.path.exists(REF_DIGESTS) else {}
        self.seen = {}

    def call(self, fn):
        """fn() on the live reference; None where the reference is not built."""
        return fn() if self.live else None

    def same(self, key: str, ref_fn, value) -> bool:
        """Is the reference's result (ref_fn(), called only on the live reference) bit for bit ``value``?"""
        if not self.live:
            assert key in self.stored, "no stored reference result %s / %s" % (self.case, key)
            return self.stored[key] == digest(value)
        x = ref_fn()
        if self.record:
            self.seen[key] = digest(x)
        else:
            assert self.stored.get(key, digest(x)) == digest(x), \
                "%s: %s differs from the stored reference digest" % (self.case, key)
        return x == value if isinstance(x, bytes) else bool(np.array_equal(x, value))

    def save(self):
        if not self.record:
            return
        db = json.load(open(REF_DIGESTS)) if os.path.exists(REF_DIGESTS) else {}
        db[self.case] = self.seen
        with open(REF_DIGESTS, "w") as f:
            json.dump(db, f, indent=0, sort_keys=True)
            f.write("\n")


def ref_lib():
    global _ref
    if _ref is None:
        L = C.CDLL(REF_SO)
        L.ref_new.restype = C.c_void_p
        L.ref_new.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_int]
        L.ref_free.argtypes = [C.c_void_p]
        L.ref_set_interp_only.argtypes = [C.c_void_p, C.c_int]
        L.ref_silence.argtypes = [C.c_int]
        L.ref_load_file.argtypes = [C.c_void_p]
        L.ref_load_raw.argtypes = [C.c_void_p, C.c_int, C.c_double, _fp, _fp, _dp]
        for f in ("ref_interp_input", "ref_interp_output", "ref_write_output"):
            getattr(L, f).argtypes = [C.c_void_p]
        L.ref_sweep.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.ref_sweep_flags.argtypes = [C.c_void_p, C.c_int, _dp, _dp, C.POINTER(C.c_ubyte), C.c_int]
        L.ref_get_vec.argtypes = [C.c_void_p, C.c_char_p, C.c_int, _dp, C.c_int]
        L.ref_mvc_per_sample.argtypes = [C.c_void_p, C.c_double, _dp, C.c_int]
        L.ref_get_scalar.argtypes = [C.c_void_p, C.c_char_p]
        L.ref_get_scalar.restype = C.c_double
        L.ref_get_cfg.argtypes = [C.c_void_p, C.POINTER(BatotpCfg)]
        L.ref_batch_run.restype = C.c_double
        L.ref_batch_run.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_double, _fp, _fp, C.c_int,
                                    _dp, _ip, _ip, _ip, _ip, _fp, C.c_int]
        _ref = L
    return _ref


class _Base:
    _pre = ""

    def vec(self, name: str, idx: int = 0) -> np.ndarray:
        g = getattr(self.L, self._pre + "_get_vec")
        n = g(self.h, name.encode(), idx, None, 0)
        if n < 0:
            raise KeyError(name)
        out = np.zeros(max(n, 1), dtype=np.float64)
        g(self.h, name.encode(), idx, out.ctypes.data_as(_dp), n)
        return out[:n]

    def scalar(self, name: str) -> float:
        return getattr(self.L, self._pre + "_get_scalar")(self.h, name.encode())

    def rows(self, name: str, n: int) -> np.ndarray:
        return np.stack([self.vec(name, j) for j in range(n)])


class Oracle(_Base):
    _pre = "orc"

    def __init__(self, cfg: BatotpCfg):
        self.L = orc_lib()
        self.cfg = cfg.copy()
        self.h = self.L.orc_new(C.byref(self.cfg))

    def __del__(self):
        if getattr(self, "h", None):
            self.L.orc_free(self.h)
            self.h = None

    def load_raw(self, n0, tres, theta=None, cart=None, timestamp=None):
        if (theta is not None and theta.dtype == np.float64) or (cart is not None and cart.dtype == np.float64):
            th = None if theta is None else np.ascontiguousarray(theta, dtype=np.float64)
            ca = None if cart is None else np.ascontiguousarray(cart, dtype=np.float64)
            ts = None if timestamp is None else np.ascontiguousarray(timestamp, dtype=np.float64)
            return self.L.orc_load_raw_f64(self.h, n0, tres, _ptr(th, _dp), _ptr(ca, _dp), _ptr(ts, _dp))
        th = None if theta is None else np.ascontiguousarray(theta, dtype=np.float32)
        ca = None if cart is None else np.ascontiguousarray(cart, dtype=np.float32)
        ts = None if timestamp is None else np.ascontiguousarray(timestamp, dtype=np.float64)
        return self.L.orc_load_raw(self.h, n0, tres, _ptr(th, _fp), _ptr(ca, _fp), _ptr(ts, _dp))

    def set_dyn_callback(self, fn):
        """fn: address of an orc_dyn_fn (e.g. dyn_fn_address("orc_demo_dyn_serial"))."""
        self.L.orc_set_dyn_callback(self.h, C.cast(fn, C.c_void_p), None)

    def interp_input(self):
        return self.L.orc_interp_input(self.h)

    def sweep(self, d, last):
        return self.L.orc_sweep(self.h, d, last)

    def interp_output(self):
        return self.L.orc_interp_output(self.h)

    def optimize(self):
        return self.L.orc_optimize(self.h)

    def mvc_per_sample(self, sdot_start: float) -> np.ndarray:
        n = int(self.scalar("nPtsC"))
        out = np.zeros(n, dtype=np.float64)
        self.L.orc_mvc_per_sample(self.h, sdot_start, out.ctypes.data_as(_dp), n)
        return out

    def pack_traj_out(self) -> bytes:
        n = self.L.orc_pack_traj_out(self.h, None, 0)
        b = C.create_string_buffer(n)
        self.L.orc_pack_traj_out(self.h, b, n)
        return b.raw

    def pack_s_sdot(self) -> bytes:
        n = self.L.orc_pack_s_sdot(self.h, None, 0)
        b = C.create_string_buffer(n)
        self.L.orc_pack_s_sdot(self.h, b, n)
        return b.raw


class Ref(_Base):
    _pre = "ref"

    def __init__(self, config_path: str, input_folder: str = "./", output_folder: str = "./",
                 auto_integ_res: bool = False, silent: bool = True):
        self.L = ref_lib()
        self.silent = silent
        if silent:
            self.L.ref_silence(1)
        self.h = self.L.ref_new(config_path.encode(), input_folder.encode(), output_folder.encode(),
                                int(auto_integ_res))
        if silent:
            self.L.ref_silence(0)
        if not self.h:
            raise RuntimeError("reference readConfigData failed for " + config_path)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.ref_free(self.h)
            self.h = None

    def set_interp_only(self, on: bool):
        self.L.ref_set_interp_only(self.h, int(on))

    def _call(self, f, *a):
        if self.silent:
            self.L.ref_silence(1)
        try:
            return f(self.h, *a)
        finally:
            if self.silent:
                self.L.ref_silence(0)

    def cfg(self) -> BatotpCfg:
        c = BatotpCfg()
        self.L.ref_get_cfg(self.h, C.byref(c))
        return c

    def load_file(self):
        return self._call(self.L.ref_load_file)

    def load_raw(self, n0, tres, theta=None, cart=None, timestamp=None):
        th = None if theta is None else np.ascontiguousarray(theta, dtype=np.float32)
        ca = None if cart is None else np.ascontiguousarray(cart, dtype=np.float32)
        ts = None if timestamp is None else np.ascontiguousarray(timestamp, dtype=np.float64)
        return self.L.ref_load_raw(self.h, n0, tres, _ptr(th, _fp), _ptr(ca, _fp), _ptr(ts, _dp))

    def interp_input(self):
        return self._call(self.L.ref_interp_input)

    def sweep(self, d, last):
        return self._call(self.L.ref_sweep, d, last)

    def sweep_flags(self, d, cap=200000):
        s = np.zeros(cap)
        sd = np.zeros(cap)
        fl = np.zeros(cap, dtype=np.uint8)
        n = self._call(self.L.ref_sweep_flags, d, s.ctypes.data_as(_dp), sd.ctypes.data_as(_dp),
                       fl.ctypes.data_as(C.POINTER(C.c_ubyte)), cap)
        return s[:n], sd[:n], fl[:n]

    def interp_output(self):
        return self._call(self.L.ref_interp_output)

    def mvc_per_sample(self, sdot_start: float) -> np.ndarray:
        n = int(self.scalar("nPtsC"))
        out = np.zeros(n, dtype=np.float64)
        self._call(self.L.ref_mvc_per_sample, sdot_start, out.ctypes.data_as(_dp), n)
        return out

    def write_output(self):
        return self._call(self.L.ref_write_output)
