#!/usr/bin/env python
"""bench.py — trajectories/s of the BA time-optimisation path on B200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's CPU implementation on the host cores
    python bench.py --workload kuka|cspr ...  # BASELINE configs[2] / configs[3] (defaults: 4096 / 65536 paths)
    python bench.py --total 1048576 ...       # strong scaling: the 2^20-path batch split over the ranks
    python bench.py --dump-outputs DIR ...    # also write the last timed step's results as DIR/*.npy (rank 0)

Workloads (seeded synthetic paths, batotp_b200/synth.py; recipes of the reference's own Octave generators):
  gen7dof (default)  configs[4]: GEN7DOF, 20 knots U[0,5]^7 -> 400 pts, joint velocity / acceleration limits;
                     `--batch` paths per GPU (default 131072 = the 2^20-path configuration at 8 GPUs, weak scaling)
  kuka               configs[2]: KUKA-LWR-IV, 4096 paths, joint + Cartesian limits through the forward kinematics,
                     strict trigonometry on the device (bit-identical port of the host libm)
  cspr               configs[3]: CSPR3DOF, 65536 paths inside the static workspace, cable-tension limits
A "step" is one pass interpInputData -> sweep(rev) -> sweep(fwd) -> interpOutputData over the batch.

value : inputs already resident in HBM, per-trajectory scalars read back, device time by CUDA events
        on the library's stream, max over ranks.
e2e   : the same metric through the C-ABI call with pinned HOST buffers, host->device copy of the
        float32 paths and device->host copy of the float32 output trajectories inside the timed region.
roofline : FP64 (the path is scalar FP64, no tensor cores): algorithmic flops of the sweep kernel
        (SURVEY §8d counting, from the kernel's own call counters) / its CUDA-event time, against the
        FP64 peak measured on this device by a DFMA micro-kernel (MEASURED_PEAKS.json has none); full-wave and
        partial (tail) launches are reported separately.
cpu_baseline : oracle/_ref (the unmodified reference, "reference") or the oracle port ("port") on the
        host cores, one trajectory per thread, on a bounded sample.
latency : single-path milliseconds (configs[0] RR stock, configs[1] UR5 at fine discretisation) through the
        same C-ABI, beside the CPU implementation on one core.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "trajectories/s"
GOLD = os.path.join(ROOT, "tests", "golden")

WORKLOADS = {
    "gen7dof": dict(cfg="GEN7DOF_config.dat", gen="gen7dof_paths", batch=131072, cart=False,
                    metric="trajectories/sec (GEN7DOF batch)",
                    text="GEN7DOF synthetic spline paths (generateGEN7DOFpath.m recipe: 20 knots U[0,5]^7 -> not-a-knot "
                         "spline -> 400 pts, seeded), stock GEN7DOF config.dat (joint vel 5 / acc 10 limits, integRes "
                         "0.01, outRes 0.008, outSmoothFact 5)"),
    "kuka": dict(cfg="KUKA_config.dat", gen="kuka_paths", batch=4096, cart=False,
                 metric="trajectories/sec (KUKA-LWR-IV batch)",
                 text="KUKA-LWR-IV synthetic spline paths (20 knots U[-0.8,0.8] x joint range -> 400 pts, tres 0.5, seeded), "
                      "stock KUKA config.dat (joint vel/acc + Cartesian velocity limit through fwdKinKuka, integRes 0.005), "
                      "strict trigonometry on the device"),
    "cspr": dict(cfg="CSPR3DOF_config.dat", gen="cspr_paths", batch=65536, cart=True,
                 metric="trajectories/sec (CSPR3DOF batch)",
                 text="CSPR3DOF synthetic Cartesian spline paths (generatePathPointsCSPR.m recipe: 20 knots -> 3801 pts, "
                      "seeded, redrawn until inside the static workspace), stock CSPR config.dat (cable tensions in "
                      "[1,12] N through dynCSPR3DOF + Par2Ser, joint + Cartesian velocity limits, integRes 0.01)"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="gen7dof", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="paths per GPU per step (0 = the workload's default)")
    ap.add_argument("--total", type=int, default=0,
                    help="strong scaling: total paths per step, split into contiguous slices over the ranks")
    ap.add_argument("--chunk", type=int, default=0,
                    help="paths resident per device pass (input interp + sweeps); 0 = the library's automatic split")
    ap.add_argument("--out-chunk", type=int, default=8192, help="paths per output-interpolation pass")
    ap.add_argument("--sweep-kernel", type=int, default=0, help="0 automatic, 1 lane per trajectory, 2 group per trajectory")
    ap.add_argument("--pipeline", type=int, default=0,
                    help="two-context chunk pipeline: 0 off (default: measured slower, see DESIGN.md), 1 automatic, "
                         "n > 1 chunks of n paths (tuning)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of the baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true", help="skip the single-path latency block")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only: skip the host-buffer leg")
    ap.add_argument("--pitched", action="store_true",
                    help="e2e leg: rows at the pitch of the longest trajectory instead of the ragged layout")
    ap.add_argument("--lib", default=None, help="experiments only: alternative build of libbatotp_cuda.so")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (rank 0, at most "
                         "64 MB): the resident leg's per-trajectory values and the host-buffer leg's output rows of a "
                         "fixed sample of trajectories, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs: only the b200 arm returns outputs")
    return args


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.f.read().splitlines():
            t = [x.strip() for x in ln.split(",")]
            if len(t) < 6:
                continue
            try:
                sm.append(float(t[0]))
                mx.append(float(t[1]))
            except ValueError:
                continue
            for nm, v in zip(names, t[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out["sm_mhz"] = statistics.median(sm)
            out["sm_max_mhz"] = max(mx)
        out["reasons"] = sorted(reasons)
        return out


# ----------------------------------------------------------------------------- workload helpers
def cpu_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def gen_paths(wl, first, count, slab=4096):
    """-> (tres, payload f32 [count, rows, n0])"""
    from batotp_b200 import synth
    gen = getattr(synth, WORKLOADS[wl]["gen"])
    parts, tres = [], None
    for at in range(0, count, slab):
        tres, p = gen(first + at, min(slab, count - at))
        parts.append(p)
    return tres, (parts[0] if len(parts) == 1 else np.concatenate(parts, axis=0))


def flops_model(cfg):
    """SURVEY §8d counting (1 flop per FP64 add/sub/mul/div/sqrt): per-call flops of A5 evalSplinePartials,
    A4 verifySecondOrderConstraints, A2 sdotLim, and the RK combine per step."""
    J = cfg.n_joints
    cart_on = bool(cfg.is_cart_vel_on or cfg.is_cart_acc_on)
    C_rows = 7 if (cfg.n_cart == 6 and cfg.path_type in (2, 3)) else max(cfg.n_cart, 3)
    a5 = 5 + 18 * J + ((18 * C_rows + 16) if cart_on else 0) + ((1 + 24 * J) if cfg.is_trq_on else 0)
    a4 = 2 + (8 * J if cfg.is_trq_on else 0) + (7 * J if cfg.is_jnt_acc_on else 0) + (16 if cfg.is_cart_acc_on else 0)
    a2 = 4 + 2 * J + (3 if cfg.is_cart_vel_on else 0)
    return dict(a5=a5, a4=a4, a2=a2, rk=110)


def bind_to_local_cpus(local, world):
    """Keeps this rank's host threads (and the first touch of its pinned buffers) on the CPUs next to its GPU;
    ranks that share one CPU list each take their own slice of it."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        txt = open("/sys/bus/pci/devices/%s/local_cpulist" % bus).read().strip()
        cpus = []
        for part in txt.split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return None
        if world > 1 and len(allowed) >= world:
            per = len(allowed) // world
            allowed = allowed[local * per:(local + 1) * per]
        os.sched_setaffinity(0, allowed)
        node = open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip()
        return dict(cpus="%d-%d" % (allowed[0], allowed[-1]) if allowed else "", count=len(allowed), numa_node=node)
    except Exception:
        return None


def cpu_runner(wl):
    """-> (kind, callable(payload f32, tres, threads) -> seconds)  (the checker libraries, used here
    only as the timed CPU baseline)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle as O
    from batotp_b200.config import read_config
    fp, ip = C.POINTER(C.c_float), C.POINTER(C.c_int)
    cfgp = os.path.join(GOLD, "synthetic", WORKLOADS[wl]["cfg"])
    cart = WORKLOADS[wl]["cart"]
    if O.ref_available():
        L = O.ref_lib()

        def run(pay, tres, nth):
            B = pay.shape[0]
            st = np.zeros(B, np.int32)
            ptr = pay.ctypes.data_as(fp)
            return L.ref_batch_run(cfgp.encode(), B, pay.shape[2], tres, None if cart else ptr, ptr if cart else None,
                                   nth, None, None, None, None, st.ctypes.data_as(ip), None, 0)
        return "reference", run
    L = O.orc_lib()
    cfg, _ = read_config(cfgp)

    def run(pay, tres, nth):
        B = pay.shape[0]
        st = np.zeros(B, np.int32)
        ptr = pay.ctypes.data_as(fp)
        return L.orc_batch_run(C.byref(cfg), B, pay.shape[2], tres, None if cart else ptr, ptr if cart else None,
                               nth, None, None, None, None, st.ctypes.data_as(ip), None, 0)
    return "port", run


def cpu_sample_rate(wl, payload, tres, seconds):
    """Times the CPU implementation on a bounded prefix of the workload. -> dict"""
    kind, run = cpu_runner(wl)
    nth = cpu_threads()
    pilot = min(payload.shape[0], 4 * nth)
    t = run(payload[:pilot], tres, nth)
    rate = pilot / max(t, 1e-9)
    n = int(min(payload.shape[0], max(pilot, rate * seconds)))
    t = run(payload[:n], tres, nth)
    return dict(value=n / t, unit=UNIT, cores=nth, kind=kind,
                sample="first %d of the step's paths, %.1f s, interpInputData+2 sweeps+interpOutputData, "
                       "one trajectory per thread" % (n, t))


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = args.workload
    kind, run = cpu_runner(wl)
    nth = cpu_threads()
    batch = args.total or (args.batch or WORKLOADS[wl]["batch"])
    # bounded sample per step: sized from a pilot so that (steps+warmup) steps stay within minutes
    tres, pilot = gen_paths(wl, 0, 4 * nth)
    t = run(pilot, tres, nth)
    rate = pilot.shape[0] / max(t, 1e-9)
    per_step = int(max(4 * nth, min(batch, rate * max(2.0, 90.0 / (args.steps + args.warmup)))))
    tres, payload = gen_paths(wl, 0, per_step)
    for _ in range(args.warmup):
        run(payload, tres, nth)
    t0 = time.time()
    tot = 0.0
    for _ in range(args.steps):
        tot += run(payload, tres, nth)
    wall = time.time() - t0
    value = per_step * args.steps / tot
    line = dict(metric=WORKLOADS[wl]["metric"], value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * tot / args.steps, higher_is_better=True,
                scaling="strong" if args.total else "weak", vs_baseline=None,
                dtype="f64", data="synthetic", impl="reference",
                config=dict(workload=WORKLOADS[wl]["text"], paths_per_step=per_step,
                            note="bounded sample of the b200 arm's workload; CPU only, rank 0"),
                cpu_baseline=dict(value=value, unit=UNIT, cores=nth, kind=kind,
                                  sample="%d paths per step, %d timed steps, wall %.1f s" % (per_step, args.steps, wall)),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    emit_line(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------- single-path latency
def latency_block(ctx):
    """configs[0] (RR stock) and configs[1] (UR5 at fine discretisation): one path through the C-ABI (host buffers in,
    float32 rows out; the group-per-trajectory sweep kernel serves a lone path) beside the CPU implementation on one
    core.  Median of 5 calls after 2."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _parity as P
    from batotp_b200 import native
    out = {}
    for key, name, fine in (("rr_stock_ms", "RR", False), ("ur5_fine_ms", "UR5", True)):
        cfg, tres, th, ca, ts = P.load_stock(name)
        cfg = cfg.copy()
        if fine:
            cfg.integ_res = 0.001
            cfg.theta_norm_res, cfg.theta_norm_res2 = cfg.theta_norm_res / 10, cfg.theta_norm_res2 / 10
            cfg.cart_norm_res, cfg.cart_norm_res2 = cfg.cart_norm_res / 10, cfg.cart_norm_res2 / 10
            cfg.out_res = 0.001
        bi = ctx.make_in(th, ca, tres, timestamp=ts)
        res = native.BatchResult(1, cfg.n_joints, cfg.n_cart, 16384, 16384, bool(cfg.is_trq_on))
        ts_ms = []
        for k in range(7):
            t0 = time.perf_counter()
            ctx.optimize_batch(cfg, bi, res)
            ts_ms.append((time.perf_counter() - t0) * 1e3)
        entry = dict(b200=statistics.median(ts_ms[2:]), rk_steps=[int(res.n_rev[0]), int(res.n_fwd[0])])
        try:
            cpu = []
            for k in range(3):
                t0 = time.perf_counter()
                P.OracleRun(cfg, tres, None if th is None else th[0], None if ca is None else ca[0],
                            None if ts is None else ts[0])
                cpu.append((time.perf_counter() - t0) * 1e3)
            entry["cpu_one_core"] = min(cpu)
            entry["cpu_kind"] = "port"
        except Exception as e:
            entry["cpu_one_core"] = None
            entry["cpu_kind"] = "unavailable: %s" % e
        out[key] = entry
    out["note"] = ("one path has no batch parallelism: 8 (RR: 4) lanes of one warp carry it through ~10^4 sequential "
                   "RK stages; wall time of the whole C-ABI call incl. copies")
    return out


# ----------------------------------------------------------------------------- output dump
DUMP_BYTES = 64_000_000
SCALARS = ("status", "n_rev", "n_fwd", "n_out", "n_cart_out", "n_grid", "t_total", "t_rev", "s_last_sec", "out_sres")


def dump_outputs(d, res_s, res_e, e2e_first):
    """--dump-outputs: the arrays the timed legs returned in their last step, as .npy files in d.
    Per-trajectory values of the resident leg (float64, exact for the integer ones) for every trajectory of the batch,
    or for a seeded sample when the batch is too large; traj_index.npy holds the trajectory indices.  Output rows of
    the host-buffer leg (float32, as returned): the trajectories res_e holds (those from e2e_first on), taken in a
    seeded order for as long as the total stays within DUMP_BYTES; each of theta_out / trq_out / cart_out is the
    concatenation of the sampled trajectories' [rows, n] blocks; rows_index.npy holds their trajectory indices,
    rows_n.npy their n (cart_n.npy that of the Cartesian blocks)."""
    os.makedirs(d, exist_ok=True)
    B = res_s.B
    per_traj = 8 * (len(SCALARS) + 1)
    idx = np.arange(B)
    if B * per_traj > DUMP_BYTES // 2:
        idx = np.sort(np.random.default_rng(1).permutation(B)[:DUMP_BYTES // 2 // per_traj])
    np.save(os.path.join(d, "traj_index.npy"), idx.astype(np.float64))
    for nm in SCALARS:
        np.save(os.path.join(d, nm + ".npy"), getattr(res_s, nm)[idx].astype(np.float64))
    if res_e is None:
        return
    left = DUMP_BYTES - per_traj * len(idx) - (1 << 16)  # (1 << 16: the .npy headers)
    names = [nm for nm in ("theta_out", "trq_out", "cart_out") if getattr(res_e, nm) is not None]
    rows = {nm: [] for nm in names + ["rows_index", "rows_n"] + (["cart_n"] if "cart_out" in names else [])}
    for b in np.random.default_rng(2).permutation(B - e2e_first):
        blk = {nm: res_e.rows(b, nm) for nm in names if nm != "cart_out"}
        if "cart_out" in names:
            blk["cart_out"] = res_e.cart_out[b, :res_e.Cin, :int(res_e.n_cart_out[b])]
        cost = sum(a.nbytes for a in blk.values()) + 24
        if cost > left:
            break
        left -= cost
        for nm, a in blk.items():
            rows[nm].append(a.ravel())
        rows["rows_index"].append([e2e_first + b])
        rows["rows_n"].append([blk["theta_out"].shape[1]])
        if "cart_out" in blk:
            rows["cart_n"].append([blk["cart_out"].shape[1]])
    for nm, parts in rows.items():
        a = np.concatenate(parts) if parts else np.zeros(0, np.float32)
        np.save(os.path.join(d, nm + ".npy"), a if nm in names else a.astype(np.float64))


# ----------------------------------------------------------------------------- B200 arm
def main_b200(args):
    import torch
    import torch.distributed as dist
    from batotp_b200 import native
    from batotp_b200.config import read_config

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the b200 arm has no CPU fallback)")
    torch.cuda.set_device(local)
    all_cpus = os.sched_getaffinity(0)
    affinity = bind_to_local_cpus(local, world)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    wl = args.workload
    W = WORKLOADS[wl]
    cfg, _ = read_config(os.path.join(GOLD, "synthetic", W["cfg"]))
    if args.total:
        total = args.total
        lo, hi = rank * total // world, (rank + 1) * total // world  # contiguous slices
        B, first = hi - lo, lo
        scaling = "strong"
    else:
        B = args.batch or W["batch"]
        total, first = world * B, rank * B
        scaling = "weak"
    J = cfg.n_joints
    tres, payload = gen_paths(wl, first, B)
    n0 = payload.shape[2]
    h_pay = torch.from_numpy(payload).pin_memory()
    d_pay = h_pay.cuda()
    ctx = native.Context(local, args.lib)
    ctx.set_chunk(args.chunk)
    ctx.set_out_chunk(args.out_chunk)
    ctx.set_sweep_kernel(args.sweep_kernel)
    ctx.set_pipeline(args.pipeline)
    peak_fma, peak_nofma = ctx.fp64_peak()
    trig_bad, trig_variant = ctx.selftest_trig(1, 1 << 20)  # the strict trigonometry reproduces this host's libm

    # ---- value: inputs resident in HBM, scalars back --------------------------------
    dp = dict(theta=None if W["cart"] else d_pay.data_ptr(), cart=d_pay.data_ptr() if W["cart"] else None, B=B, n0_max=n0)
    bi_dev = ctx.make_in(tres=tres, device_ptrs=dp)
    res_s = native.BatchResult(B, J, cfg.n_cart, 0, 0, bool(cfg.is_trq_on), want_rows=False, want_hist=False)

    def step_resident():
        ctx.optimize_batch(cfg, bi_dev, res_s)

    for _ in range(args.warmup):
        step_resident()
    barrier()
    ctx.stats_reset()
    clk = ClockSampler(local)
    try:  # the sampler is a child process: it must not outlive a failed step
        ctx.timer_start()
        for _ in range(args.steps):
            step_resident()
        ms = ctx.timer_stop_ms()
        barrier()
    finally:
        clocks = clk.stop()
    st = ctx.stats()
    slog = ctx.sweep_log()
    ms = max_over_ranks(ms)
    ok = int((res_s.status & native.ST_FATAL_MASK == 0).sum())
    value = total * args.steps / (ms * 1e-3)

    # ---- roofline of the dominant kernel (the sweeps) ---------------------------------
    fm = flops_model(cfg)
    steps_rk, ver, ntraj = st["steps"], st["verifies"], max(st["trajectories"], 1)
    n_eval = 6 * steps_rk + 4 * ntraj           # evalSplinePartials calls (A5): 6/step + 2 per sweep prologue
    n_lim = 7 * steps_rk + 4 * ntraj            # sdotLim calls (A2)
    flops = n_eval * fm["a5"] + ver * fm["a4"] + n_lim * fm["a2"] + fm["rk"] * steps_rk
    sweep_s = st["sweep_ms"] * 1e-3
    achieved = flops / max(sweep_s, 1e-12) * 1e-12
    flops_per_traj = flops / ntraj
    # full-wave launches (the largest chunk size seen) and partial ones (tail chunks, stragglers) separately
    launches = {}
    if slog:
        full_b = max(b for _, b, _ in slog)
        for nm, sel in (("full_wave", [r for r in slog if r[1] == full_b]), ("partial", [r for r in slog if r[1] != full_b])):
            if sel:
                t_ms = sum(r[0] for r in sel)
                n_tr = sum(r[1] for r in sel)
                tf = flops_per_traj * n_tr / (t_ms * 1e-3) * 1e-12
                launches[nm] = dict(launches=len(sel), paths_per_launch=n_tr / len(sel), avg_launch_ms=t_ms / len(sel),
                                    achieved=tf, frac=tf / max(peak_fma, 1e-12),
                                    kernel={1: "k_sweep", 2: "k_sweep_group"}[sel[0][2]])
    # DRAM traffic of the sweep kernel: from this round's ncu --set full capture (profiles/), per path, scaled to the
    # paths per launch of this run; null when the capture is of another workload
    traffic, traffic_src = None, None
    try:
        import csv
        prof = os.path.join(ROOT, "profiles", "r2_sweep_ncu_full_summary_%s.csv" % wl)
        vals = {r[0]: (r[1], float(r[2])) for r in csv.reader(open(prof)) if len(r) >= 3 and not r[0].startswith("#")
                and r[0] != "metric"}
        gb = sum(v * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[u]
                 for k, (u, v) in vals.items() if k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
        cap_paths = vals["paths_in_captured_launch"][1]
        traffic = gb / cap_paths * (ntraj / max(st["sweep_launches"], 1))
        traffic_src = ("profiles/%s (dram__bytes_read+write of a %d-path launch of this round's kernel, per path)"
                       % (os.path.basename(prof), int(cap_paths)))
    except Exception:
        pass
    kern_names = sorted({{1: "k_sweep", 2: "k_sweep_group"}[r[2]] for r in slog}) if slog else ["k_sweep"]
    roof = dict(bound="fp64", achieved=achieved, peak=peak_fma, unit="TFLOP/s", frac=achieved / max(peak_fma, 1e-12),
                traffic=traffic, traffic_unit="bytes per launch", traffic_source=traffic_src,
                kernel="+".join(kern_names), launches=st["sweep_launches"],
                avg_launch_ms=st["sweep_ms"] / max(st["sweep_launches"], 1), by_launch_kind=launches,
                peak_source="measured in this run (DFMA chains); MEASURED_PEAKS.json has no FP64 entry",
                peak_nofma=peak_nofma, frac_of_nofma_peak=achieved / max(peak_nofma, 1e-12),
                flops_per_trajectory=flops_per_traj, share_of_step=sweep_s / max(ms * 1e-3, 1e-12),
                share_note="sum of the sweep launches' own durations / step time; a tail chunk's launch runs beside "
                           "other kernels (tail overlap), so with a tail this exceeds the sweep's share of the timeline",
                counting="SURVEY 8d: 1 flop per FP64 add/sub/mul/div/sqrt; A5=%d, A4=%d, A2=%d per call, RK=110/step"
                         % (fm["a5"], fm["a4"], fm["a2"]))
    launches_value = st["launches"]

    # ---- e2e: pinned host inputs in, float32 trajectories out --------------------------------------
    # One C-ABI call per step over the rank's whole batch: inside it the library moves chunk k+1's rows to the
    # device and chunk k's results to the host while it computes.  The result buffer is pinned and reused; rows
    # use the pitch of the longest trajectory (known from the resident leg).
    out_cap = int(res_s.n_out.max()) if ok else 4096
    h_np = h_pay.numpy()
    want_cart = cfg.n_cart > 0 and wl != "gen7dof"  # a generic robot has no Cartesian data: its rows are zeros
    # ragged layout (the default where no Cartesian rows travel): every trajectory's [J][n_out] block at its own
    # length, so no padding crosses the host link; the capacity is the sum of the lengths (known from the resident leg)
    ragged = not args.pitched and not want_cart
    rag_cap = int(res_s.n_out.astype(np.int64).sum()) + 1024
    sl = B
    res_e = None
    while res_e is None:
        try:
            if ragged:
                res_e = native.BatchResult(sl, J, 0, 0, 0, bool(cfg.is_trq_on), want_rows=True, want_hist=False,
                                           pinned=True, ragged_cap=rag_cap)
            else:
                res_e = native.BatchResult(sl, J, cfg.n_cart if want_cart else 0, out_cap, 0, bool(cfg.is_trq_on),
                                           want_rows=True, want_hist=False, pinned=True)
        except Exception:
            if sl <= 1024 or ragged:
                raise
            sl = (sl + 1) // 2

    def step_e2e():
        chk = 0.0
        for at in range(0, B, sl):
            n = min(sl, B - at)
            bi = ctx.make_in(theta=None if W["cart"] else h_np[at:at + n], cart=h_np[at:at + n] if W["cart"] else None,
                             tres=tres)
            ctx.optimize_batch(cfg, bi, res_e)
            chk += float(res_e.t_total[:n].sum())
        return chk

    e2e = None
    if not args.skip_e2e:
        for _ in range(max(1, min(args.warmup, 2))):
            step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
        torch.cuda.synchronize()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        nsl = (B + sl - 1) // sl
        if ragged:
            rows_b = int(res_s.n_out.astype(np.int64).sum()) * J * 4 * (2 if cfg.is_trq_on else 1)
            d2h_b = rows_b + sum(getattr(res_e, nm).nbytes for nm in ("status", "n_rev", "n_fwd", "n_out", "n_cart_out",
                                                                       "n_grid", "t_total", "t_rev", "s_last_sec", "out_sres"))
        else:
            d2h_b = nsl * res_e.d2h_bytes()
        e2e = dict(value=total * args.steps / e2e_s, unit=UNIT, h2d_bytes_per_step=int(payload.nbytes),
                   d2h_bytes_per_step=int(d2h_b),
                   note="C-ABI batotp_cuda_optimize_batch on pinned host buffers, %d call(s) of %d paths per step per rank; "
                        "float32 rows (%s) + per-trajectory scalars copied back; bytes per rank"
                        % (nsl, sl, "ragged: every trajectory at its own length, the payload of trajWriteBIN" if ragged
                           else "pitch %d points = the longest trajectory" % out_cap))

    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res_s, None if e2e is None else res_e, (B - 1) // sl * sl)

    line = None
    if rank == 0:
        lat = None
        if not args.no_latency:
            try:
                lat = latency_block(ctx)
            except Exception as e:
                lat = dict(error=str(e))
        line = dict(metric=W["metric"], value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling=scaling, vs_baseline=None,
                    dtype="f64", data="synthetic",
                    config=dict(workload=W["text"], paths_per_gpu=B, paths_total=total,
                                sweep_kernel={0: "automatic", 1: "lane", 2: "group"}[args.sweep_kernel],
                                pipeline={0: "off", 1: "automatic"}.get(args.pipeline, "chunks of %d" % args.pipeline),
                                parallelism="independent contiguous slices per GPU, no collective",
                                l2="inputs (%.0f MB/GPU) and per-chunk tables exceed the 126 MB L2" % (payload.nbytes / 1e6),
                                optimised=ok, mean_rk_steps=steps_rk / ntraj,
                                mean_verifies_per_stage=ver / max(6 * steps_rk, 1),
                                strict_trig=dict(variant=trig_variant, mismatches_vs_host_libm=trig_bad, checked=2 << 20),
                                host_affinity=affinity),
                    clocks=clocks, e2e=e2e, gpu_launches=int(launches_value), roofline=roof, latency=lat)
        if not args.no_cpu_baseline and world == 1:  # (rank 0 at N = 1 only: the CPU leg wants every host core)
            try:
                os.sched_setaffinity(0, all_cpus)
                line["cpu_baseline"] = cpu_sample_rate(wl, payload, tres, args.cpu_seconds)
            except Exception as e:  # the checker libraries are optional at bench time
                line["cpu_baseline"] = dict(value=None, unit=UNIT, cores=cpu_threads(), kind="unavailable", sample=str(e))
        emit_line(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()
    return 0


_REAL_STDOUT = None


def emit_line(text):
    """The one JSON line of this process, on the real stdout (see main)."""
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        print(text, flush=True)
        return
    os.write(_REAL_STDOUT, (text + "\n").encode())


def main():
    global _REAL_STDOUT
    args = parse()
    # Rank 0's stdout carries exactly one JSON line: whatever libraries print there meanwhile (NCCL's version
    # banner, for one) goes to stderr; emit_line writes to the saved descriptor.
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return main_reference(args)
    return main_b200(args)


if __name__ == "__main__":
    sys.exit(main())
