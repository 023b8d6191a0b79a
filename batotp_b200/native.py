"""ctypes binding of include/batotp_cuda.h (the C-ABI of the CUDA library).

The product library is ``batotp_b200/lib/libbatotp_cuda.so`` (built by
``__graft_entry__.build()`` with nvcc for sm_100a).  There is no CPU fallback: if the
library is missing, or no CUDA device is present, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

from .config import BatotpCfg

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libbatotp_cuda.so")

_fp = C.POINTER(C.c_float)
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_bp = C.POINTER(C.c_ubyte)

ST_FATAL_MASK = 1 | 2 | 4 | 8 | 16 | 32 | 64 | 256 | 512
ST_BISECT_FAIL = 128


class BatchIn(C.Structure):
    _fields_ = [("B", C.c_int), ("n0_max", C.c_int), ("n0", _ip), ("tres", _dp), ("tres_all", C.c_double),
                ("theta_f32", C.c_void_p), ("cart_f32", C.c_void_p), ("theta_f64", C.c_void_p),
                ("cart_f64", C.c_void_p), ("timestamp", C.c_void_p), ("on_device", C.c_int)]


class BatchOut(C.Structure):
    _fields_ = [("out_cap", C.c_int), ("hist_cap", C.c_int), ("status", _ip), ("n_rev", _ip), ("n_fwd", _ip),
                ("n_out", _ip), ("n_cart_out", _ip), ("n_grid", _ip), ("t_total", _dp), ("t_rev", _dp),
                ("s_last_sec", _dp), ("out_sres", _dp), ("theta_out", C.c_void_p), ("cart_out", C.c_void_p),
                ("trq_out", C.c_void_p), ("hist", C.c_void_p), ("flags", C.c_void_p), ("on_device", C.c_int),
                ("row_offset", C.POINTER(C.c_longlong)), ("ragged_cap", C.c_longlong)]


class NativeError(RuntimeError):
    pass


_libs = {}


def load(path: Optional[str] = None):
    """Load the C-ABI library (default: the in-tree product build).  Raises if it is missing."""
    path = path or LIB_PATH
    if path in _libs:
        return _libs[path]
    if not os.path.exists(path):
        raise NativeError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)" % path)
    L = C.CDLL(path)
    L.batotp_cuda_device_count.restype = C.c_int
    L.batotp_cuda_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.batotp_cuda_destroy.argtypes = [C.c_void_p]
    L.batotp_cuda_last_error.argtypes = [C.c_void_p]
    L.batotp_cuda_last_error.restype = C.c_char_p
    L.batotp_cuda_set_chunk.argtypes = [C.c_void_p, C.c_int]
    L.batotp_cuda_set_out_chunk.argtypes = [C.c_void_p, C.c_int]
    L.batotp_cuda_set_max_steps.argtypes = [C.c_void_p, C.c_int]
    L.batotp_cuda_set_tail_overlap.argtypes = [C.c_void_p, C.c_int]
    L.batotp_cuda_set_step_hint.argtypes = [C.c_void_p, C.c_int]
    L.batotp_cuda_set_dyn_callback.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.batotp_cuda_set_sweep_kernel.argtypes = [C.c_void_p, C.c_int]
    L.batotp_cuda_set_walker_kernel.argtypes = [C.c_void_p, C.c_int]
    L.batotp_cuda_launch_count.argtypes = [C.c_void_p]
    L.batotp_cuda_launch_count.restype = C.c_long
    L.batotp_cuda_stats.argtypes = [C.c_void_p, _dp, C.c_int]
    L.batotp_cuda_sweep_log.argtypes = [C.c_void_p, _dp, _ip, _ip, C.c_int]
    L.batotp_cuda_set_keep_f64.argtypes = [C.c_void_p, C.c_int]
    L.batotp_cuda_fp64_peak.argtypes = [C.c_void_p, _dp, _dp]
    L.batotp_cuda_selftest_div.argtypes = [C.c_void_p, C.c_ulonglong, C.c_longlong, C.POINTER(C.c_longlong),
                                           C.POINTER(C.c_longlong)]
    L.batotp_cuda_selftest_trig.argtypes = [C.c_void_p, C.c_ulonglong, C.c_longlong, C.POINTER(C.c_longlong),
                                            C.POINTER(C.c_int)]
    L.batotp_cuda_selftest_bisect.argtypes = [C.c_void_p, C.c_ulonglong, C.c_longlong, C.POINTER(C.c_longlong)]
    L.batotp_cuda_stats_reset.argtypes = [C.c_void_p]
    L.batotp_cuda_timer.argtypes = [C.c_void_p, C.c_int, _dp]
    L.batotp_cuda_set_profile.argtypes = [C.c_void_p, C.c_int]
    L.batotp_cuda_profile_dump.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    L.batotp_cuda_optimize_batch.argtypes = [C.c_void_p, C.POINTER(BatotpCfg), C.POINTER(BatchIn), C.POINTER(BatchOut)]
    L.batotp_cuda_load.argtypes = [C.c_void_p, C.POINTER(BatotpCfg), C.POINTER(BatchIn)]
    for f in ("batotp_cuda_interp_input", "batotp_cuda_sweeps", "batotp_cuda_interp_output"):
        getattr(L, f).argtypes = [C.c_void_p]
    L.batotp_cuda_fetch.argtypes = [C.c_void_p, C.POINTER(BatchOut)]
    L.batotp_cuda_mvc_per_sample.argtypes = [C.c_void_p, C.c_double, _dp, C.c_int]
    L.batotp_cuda_get_f64.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, _dp, C.c_int]
    L.batotp_writer_create.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]
    L.batotp_writer_submit.argtypes = [C.c_void_p, C.POINTER(BatotpCfg), C.POINTER(BatchOut), C.c_longlong, C.c_int,
                                       C.c_int]
    L.batotp_writer_wait.argtypes = [C.c_void_p, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    L.batotp_writer_destroy.argtypes = [C.c_void_p]
    _libs[path] = L
    return L


class Writer:
    """Batch file writer (include/batotp_cuda.h: batotp_writer_*): traj_out_<index>.dat / s-sdot_<index>.dat."""

    def __init__(self, directory: str, threads: int = 4, lib_path: Optional[str] = None):
        self.L = load(lib_path)
        h = C.c_void_p()
        if self.L.batotp_writer_create(directory.encode(), threads, C.byref(h)) != 0:
            raise NativeError("batotp_writer_create failed")
        self.h = h
        self._keep = []

    def submit(self, cfg: BatotpCfg, res: "BatchResult", base_index: int, first: int, count: int):
        self._keep.append((cfg, res))  # the arrays must outlive the write
        if self.L.batotp_writer_submit(self.h, C.byref(cfg), C.byref(res.c), base_index, first, count) != 0:
            raise NativeError("batotp_writer_submit failed")

    def wait(self):
        w, f = C.c_longlong(0), C.c_longlong(0)
        rc = self.L.batotp_writer_wait(self.h, C.byref(w), C.byref(f))
        self._keep.clear()
        return rc, w.value, f.value

    def close(self):
        if getattr(self, "h", None):
            self.L.batotp_writer_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BatchResult:
    """Host-side view of a batotp_batch_out."""

    def __init__(self, B: int, J: int, Cin: int, out_cap: int, hist_cap: int, trq: bool, want_rows=True,
                 want_hist=True, pinned=False, ragged_cap: int = 0):
        """ragged_cap > 0: ragged joint / torque rows (batotp_batch_out.row_offset): theta_out is a flat float32
        array of ragged_cap * J values, trajectory b's block is rows(b) = theta_out[row_offset[b]*J ...] viewed as
        [J, n_out[b]]; no Cartesian rows in this mode."""
        def arr(shape, dt):
            if pinned:
                import torch
                t = torch.zeros(shape, dtype={np.float32: torch.float32, np.float64: torch.float64,
                                              np.int32: torch.int32, np.int64: torch.int64, np.uint8: torch.uint8}[dt]).pin_memory()
                self._keep.append(t)
                return t.numpy()
            return np.zeros(shape, dtype=dt)

        self._keep = []
        self.B, self.J, self.Cin = B, J, Cin
        self.status = arr(B, np.int32)
        self.n_rev = arr(B, np.int32)
        self.n_fwd = arr(B, np.int32)
        self.n_out = arr(B, np.int32)
        self.n_cart_out = arr(B, np.int32)
        self.n_grid = arr(B, np.int32)
        self.t_total = arr(B, np.float64)
        self.t_rev = arr(B, np.float64)
        self.s_last_sec = arr(B, np.float64)
        self.out_sres = arr(B, np.float64)
        self.ragged_cap = int(ragged_cap)
        if ragged_cap > 0:
            self.theta_out = arr((ragged_cap * J,), np.float32)
            self.cart_out = None
            self.trq_out = arr((ragged_cap * J,), np.float32) if trq else None
            self.row_offset = arr(B, np.int64)
        else:
            self.theta_out = arr((B, J, out_cap), np.float32) if want_rows else None
            self.cart_out = arr((B, max(Cin, 1), out_cap), np.float32) if (want_rows and Cin > 0) else None
            self.trq_out = arr((B, J, out_cap), np.float32) if (want_rows and trq) else None
            self.row_offset = None
        self.hist = arr((B, 4, hist_cap), np.float32) if want_hist else None
        self.flags = arr((B, 2, hist_cap), np.uint8) if want_hist else None
        self.c = BatchOut()
        self.c.out_cap = out_cap if want_rows else 0
        self.c.hist_cap = hist_cap if want_hist else 0
        for nm, tp in (("status", _ip), ("n_rev", _ip), ("n_fwd", _ip), ("n_out", _ip), ("n_cart_out", _ip),
                       ("n_grid", _ip), ("t_total", _dp), ("t_rev", _dp), ("s_last_sec", _dp), ("out_sres", _dp)):
            setattr(self.c, nm, getattr(self, nm).ctypes.data_as(tp))
        for nm in ("theta_out", "cart_out", "trq_out", "hist", "flags"):
            a = getattr(self, nm)
            setattr(self.c, nm, a.ctypes.data if a is not None else None)
        self.c.on_device = 0
        if self.row_offset is not None:
            self.c.row_offset = self.row_offset.ctypes.data_as(C.POINTER(C.c_longlong))
            self.c.ragged_cap = self.ragged_cap
            self.c.out_cap = 0

    def rows(self, b: int, which: str = "theta_out") -> np.ndarray:
        """[J, n_out[b]] view of trajectory b's rows (either layout)."""
        a = getattr(self, which)
        n = int(self.n_out[b])
        if self.row_offset is None:
            return a[b, :, :n]
        o = int(self.row_offset[b]) * self.J
        return a[o:o + self.J * n].reshape(self.J, n)

    def d2h_bytes(self) -> int:
        n = 0
        for nm in ("status", "n_rev", "n_fwd", "n_out", "n_cart_out", "n_grid", "t_total", "t_rev", "s_last_sec",
                   "out_sres", "theta_out", "cart_out", "trq_out", "hist", "flags"):
            a = getattr(self, nm)
            if a is not None:
                n += a.nbytes
        return n


class Context:
    """One device context (include/batotp_cuda.h: batotp_cuda_create)."""

    def __init__(self, device: int = 0, lib_path: Optional[str] = None):
        self.L = load(lib_path)
        h = C.c_void_p()
        if self.L.batotp_cuda_create(device, C.byref(h)) != 0 or not h:
            raise NativeError("batotp_cuda_create(%d) failed: no usable CUDA device (no CPU fallback)" % device)
        self.h = h
        self._keep = []

    def close(self):
        if getattr(self, "h", None):
            self.L.batotp_cuda_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _err(self, what):
        raise NativeError("%s failed: %s" % (what, (self.L.batotp_cuda_last_error(self.h) or b"").decode()))

    def set_chunk(self, n: int):
        self.L.batotp_cuda_set_chunk(self.h, n)

    def set_out_chunk(self, n: int):
        self.L.batotp_cuda_set_out_chunk(self.h, n)

    def set_max_steps(self, n: int):
        self.L.batotp_cuda_set_max_steps(self.h, n)

    def set_sweep_kernel(self, mode: int):
        """0 automatic, 1 one trajectory per lane, 2 a group of lanes per trajectory."""
        self.L.batotp_cuda_set_sweep_kernel(self.h, mode)

    def set_walker_kernel(self, mode: int):
        """0 automatic, 1 one thread per trajectory, 2 point-parallel increments + a group of lanes per trajectory."""
        self.L.batotp_cuda_set_walker_kernel(self.h, mode)

    def set_pipeline(self, on: int):
        """Kept because bench.py passes --pipeline: 0 does nothing, anything else raises."""
        if int(on) != 0:
            raise NativeError("the two-context chunk pipeline was removed from the library (see DESIGN.md)")

    def set_dyn_callback(self, fn, user=None):
        """fn: address of (or ctypes pointer to) a batotp_dyn_fn; None switches it off."""
        self._dyn = fn
        self.L.batotp_cuda_set_dyn_callback(self.h, C.cast(fn, C.c_void_p) if fn is not None else None, user)

    def set_step_hint(self, n: int):
        self.L.batotp_cuda_set_step_hint(self.h, n)

    def set_tail_overlap(self, on: bool):
        self.L.batotp_cuda_set_tail_overlap(self.h, 1 if on else 0)

    def set_keep_f64(self, on: bool):
        self.L.batotp_cuda_set_keep_f64(self.h, int(on))

    def launch_count(self) -> int:
        return int(self.L.batotp_cuda_launch_count(self.h))

    def stats(self) -> dict:
        v = (C.c_double * 6)()
        self.L.batotp_cuda_stats(self.h, v, 6)
        return dict(sweep_ms=v[0], sweep_launches=int(v[1]), verifies=int(v[2]), steps=int(v[3]),
                    trajectories=int(v[4]), launches=int(v[5]))

    def sweep_log(self):
        """[(device ms, trajectories, kernel)] of the sweep launches since the last stats_reset."""
        cap = 4096
        ms, nt, kk = (C.c_double * cap)(), (C.c_int * cap)(), (C.c_int * cap)()
        n = self.L.batotp_cuda_sweep_log(self.h, ms, nt, kk, cap)
        return [(ms[i], nt[i], kk[i]) for i in range(min(n, cap))]

    def fp64_peak(self):
        a, b = C.c_double(0), C.c_double(0)
        self.L.batotp_cuda_fp64_peak(self.h, C.byref(a), C.byref(b))
        return a.value, b.value

    def selftest_div(self, seed: int, n: int):
        bad, fast = C.c_longlong(0), C.c_longlong(0)
        if self.L.batotp_cuda_selftest_div(self.h, seed, n, C.byref(bad), C.byref(fast)) != 0:
            self._err('batotp_cuda_selftest_div')
        return bad.value, fast.value

    def selftest_bisect(self, seed: int, n: int) -> int:
        bad = C.c_longlong(0)
        if self.L.batotp_cuda_selftest_bisect(self.h, seed, n, C.byref(bad)) != 0:
            self._err('batotp_cuda_selftest_bisect')
        return bad.value

    def selftest_trig(self, seed: int, n: int):
        """-> (mismatches against the host libm's sin/cos, arithmetic variant: 1 plain, 3 fused multiply-adds)"""
        bad, var = C.c_longlong(0), C.c_int(0)
        if self.L.batotp_cuda_selftest_trig(self.h, seed, n, C.byref(bad), C.byref(var)) != 0:
            self._err('batotp_cuda_selftest_trig')
        return bad.value, var.value

    def set_profile(self, on: bool):
        self.L.batotp_cuda_set_profile(self.h, int(on))

    def profile(self) -> dict:
        """{kernel: (total_ms, launches)} since set_profile(True)."""
        buf = C.create_string_buffer(1 << 16)
        self.L.batotp_cuda_profile_dump(self.h, buf, len(buf))
        out = {}
        for ln in buf.value.decode().splitlines():
            nm, ms, n = ln.rsplit(",", 2)
            out[nm] = (float(ms), int(n))
        return out

    def stats_reset(self):
        self.L.batotp_cuda_stats_reset(self.h)

    def timer_start(self):
        self.L.batotp_cuda_timer(self.h, 0, None)

    def timer_stop_ms(self) -> float:
        ms = C.c_double(0)
        self.L.batotp_cuda_timer(self.h, 1, C.byref(ms))
        return ms.value

    @staticmethod
    def make_in(theta=None, cart=None, tres=0.01, n0=None, timestamp=None, device_ptrs=None) -> BatchIn:
        """theta/cart: numpy [B, rows, n0_max] float32 or float64 (C-contiguous).
        device_ptrs: optional dict(theta=int, cart=int, B=, n0_max=, f64=bool) for HBM-resident inputs."""
        bi = BatchIn()
        keep = []
        if device_ptrs:
            bi.B, bi.n0_max = device_ptrs["B"], device_ptrs["n0_max"]
            f64 = device_ptrs.get("f64", False)
            if f64:
                bi.theta_f64, bi.cart_f64 = device_ptrs.get("theta"), device_ptrs.get("cart")
            else:
                bi.theta_f32, bi.cart_f32 = device_ptrs.get("theta"), device_ptrs.get("cart")
            bi.on_device = 1
        else:
            ref = theta if theta is not None else cart
            bi.B, bi.n0_max = ref.shape[0], ref.shape[2]
            f64 = ref.dtype == np.float64
            for nm, a in (("theta", theta), ("cart", cart)):
                if a is None:
                    continue
                assert a.flags["C_CONTIGUOUS"] and a.dtype == ref.dtype
                keep.append(a)
                setattr(bi, "%s_%s" % (nm, "f64" if f64 else "f32"), a.ctypes.data)
            bi.on_device = 0
        if np.ndim(tres) == 0:
            bi.tres_all = float(tres)
            bi.tres = None
        else:
            t = np.ascontiguousarray(tres, dtype=np.float64)
            keep.append(t)
            bi.tres = t.ctypes.data_as(_dp)
        if n0 is not None:
            n = np.ascontiguousarray(n0, dtype=np.int32)
            keep.append(n)
            bi.n0 = n.ctypes.data_as(_ip)
        if timestamp is not None:
            ts = np.ascontiguousarray(timestamp, dtype=np.float64)
            keep.append(ts)
            bi.timestamp = ts.ctypes.data
        bi._keep = keep
        return bi

    def optimize_batch(self, cfg: BatotpCfg, bi: BatchIn, res: BatchResult):
        if self.L.batotp_cuda_optimize_batch(self.h, C.byref(cfg), C.byref(bi), C.byref(res.c)) != 0:
            self._err("batotp_cuda_optimize_batch")
        return res

    # phase-wise (one resident chunk)
    def load(self, cfg: BatotpCfg, bi: BatchIn):
        self._cfg = cfg
        if self.L.batotp_cuda_load(self.h, C.byref(cfg), C.byref(bi)) != 0:
            self._err("batotp_cuda_load")

    def interp_input(self):
        if self.L.batotp_cuda_interp_input(self.h) != 0:
            self._err("batotp_cuda_interp_input")

    def sweeps(self):
        if self.L.batotp_cuda_sweeps(self.h) != 0:
            self._err("batotp_cuda_sweeps")

    def interp_output(self):
        if self.L.batotp_cuda_interp_output(self.h) != 0:
            self._err("batotp_cuda_interp_output")

    def fetch(self, res: BatchResult):
        if self.L.batotp_cuda_fetch(self.h, C.byref(res.c)) != 0:
            self._err("batotp_cuda_fetch")
        return res

    def mvc_per_sample(self, B: int, cap: int, sdot_start: float) -> np.ndarray:
        out = np.zeros((B, cap), dtype=np.float64)
        if self.L.batotp_cuda_mvc_per_sample(self.h, sdot_start, out.ctypes.data_as(_dp), cap) != 0:
            self._err("batotp_cuda_mvc_per_sample")
        return out

    def get_f64(self, name: str, traj: int, row: int = 0) -> np.ndarray:
        n = self.L.batotp_cuda_get_f64(self.h, name.encode(), traj, row, None, 0)
        if n < 0:
            raise KeyError(name)
        out = np.zeros(max(n, 1), dtype=np.float64)
        self.L.batotp_cuda_get_f64(self.h, name.encode(), traj, row, out.ctypes.data_as(_dp), n)
        return out[:n]
