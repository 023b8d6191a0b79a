"""Cost of per-trajectory limits (batotp_batch_in.limits) on the device.

For GEN7DOF x131072, KUKA x4096 and CSPR3DOF x65536 (the bench.py workloads), in alternating repeats:
  null   limits = NULL
  equal  one row per path equal to the cfg's limits (the LIM kernel instantiations, same results)
  mixed  seeded heterogeneous rows: a speed-override factor f per path, drawn from 8 values in [FMIN, 1],
         applied to the velocity limits and, squared, to the acceleration limits
and, for GEN7DOF, the mixed batch split into 8 calls, one per limit class (what a caller without the feature does).
Reports trajectories per second (host clock around the call, which ends in a device synchronise) and the per-launch
sweep times of batotp_cuda_sweep_log.  Writes one JSON file (default profiles/trajectory_limits_bench.json).

    python scripts/trajectory_limits_bench.py --repeats 3 --out /tmp/trajectory_limits_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from batotp_b200 import native  # noqa: E402
from batotp_b200.config import limit_row  # noqa: E402
import _parity as P  # noqa: E402

SIZES = {"GEN7DOF": 131072, "KUKA": 4096, "CSPR3DOF": 65536}
# smallest speed-override factor: KUKA paths take ~18 600 steps per sweep at the stock limits, and slower classes
# would reach the default step ceiling
FMIN = {"GEN7DOF": 0.4, "KUKA": 0.7, "CSPR3DOF": 0.4}
N_CLASSES = 8


def speed_rows(cfg, B, seed, fmin):
    rng = np.random.RandomState(seed)
    f = np.linspace(fmin, 1.0, N_CLASSES)
    cls = rng.randint(0, N_CLASSES, B)
    rows = np.tile(limit_row(cfg), (B, 1))
    rows[:, 0:7] *= f[cls, None]
    rows[:, 7:14] *= (f[cls] ** 2)[:, None]
    rows[:, 28] *= f[cls]
    rows[:, 29] *= f[cls] ** 2
    return rows, cls


def timed(ctx, cfg, th, ca, tres, limits, res):
    ctx.stats_reset()
    bi = ctx.make_in(th, ca, tres, limits=limits)
    t0 = time.perf_counter()
    ctx.optimize_batch(cfg, bi, res)
    dt = time.perf_counter() - t0
    st = ctx.stats()
    return dt, st["sweep_ms"], [round(x[0], 2) for x in ctx.sweep_log()]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % e
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--workloads", default="GEN7DOF,KUKA,CSPR3DOF")
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the workload sizes (rehearsal only)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "trajectory_limits_bench.json"))
    args = ap.parse_args()
    ctx = native.Context(0)
    out = dict(gpu=gpu_info(), repeats=args.repeats, results={})
    for name in args.workloads.split(","):
        B = max(1, int(SIZES[name] * args.scale))
        cfg, tres, th, ca = P.load_synth(name, 0, B)
        trq = bool(cfg.is_trq_on)
        res = native.BatchResult(B, cfg.n_joints, cfg.n_cart, 0, 0, trq, want_rows=False, want_hist=False)
        equal = np.tile(limit_row(cfg), (B, 1))
        mixed, cls = speed_rows(cfg, B, 7, FMIN[name])
        legs = {"null": None, "equal": equal, "mixed": mixed}
        rec = {k: [] for k in legs}
        if name == "GEN7DOF":
            rec["split8"] = []
        timed(ctx, cfg, th, ca, tres, None, res)  # warm-up: module load, workspaces, learnt capacities
        timed(ctx, cfg, th, ca, tres, mixed, res)
        t_null = None
        for r in range(args.repeats):
            for leg, lim in legs.items():
                dt, sw, log = timed(ctx, cfg, th, ca, tres, lim, res)
                rec[leg].append(dict(s=round(dt, 4), traj_per_s=round(B / dt, 1), sweep_ms=round(sw, 2), launches=log))
                if leg == "null":
                    t_null = res.t_total.copy()
                if leg == "equal":
                    assert np.array_equal(res.t_total, t_null), "rows equal to the cfg changed a result"
            if name == "GEN7DOF":
                tot, sw_tot, logs = 0.0, 0.0, []
                for k in range(N_CLASSES):
                    idx = np.nonzero(cls == k)[0]
                    sub = lambda a: None if a is None else np.ascontiguousarray(a[idx])  # noqa: E731
                    c = cfg.copy()
                    for i in range(7):
                        c.jnt_vel_max[i], c.jnt_acc_max[i] = mixed[idx[0], i], mixed[idx[0], 7 + i]
                    rk = native.BatchResult(len(idx), cfg.n_joints, cfg.n_cart, 0, 0, trq, want_rows=False,
                                            want_hist=False)
                    dt, sw, log = timed(ctx, c, sub(th), sub(ca), tres, None, rk)
                    tot += dt
                    sw_tot += sw
                    logs += log
                rec["split8"].append(dict(s=round(tot, 4), traj_per_s=round(B / tot, 1), sweep_ms=round(sw_tot, 2),
                                          launches=logs))
        summ = {}
        for leg, v in rec.items():
            tp = [x["traj_per_s"] for x in v]
            sw = [x["sweep_ms"] for x in v]
            summ[leg] = dict(traj_per_s_median=float(np.median(tp)), traj_per_s_min=min(tp), traj_per_s_max=max(tp),
                             sweep_ms_median=float(np.median(sw)), sweep_ms_min=min(sw), sweep_ms_max=max(sw))
        out["results"][name] = dict(paths=B, summary=summ, runs=rec)
        print(name, json.dumps(summ), flush=True)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
