"""Leave-one-out timing on the sample sets of the BASELINE configs; prints one JSON line.

    python scripts/loo_time.py [--reps 3] [--out FILE]

Per workload (C2: 1e4 samples 2-D k=20 OK; C3a: 1e5 3-D k=32 SK; C5: 1e6 3-D k=64 OK; C4: 2e4 global OK):
  * gsk_krige_loo wall time (host clock around the call, which ends in a device synchronise) and device time
    (gsk_get_timing: ms_plan + ms_total), samples/s;
  * the phases of a separate run with phase timing on (local: search of k+1 plus the self-removal, solve; global: the
    pass over L⁻¹ alone against the plan), and the self-removal kernel alone from torch.profiler in a third run;
  * for comparison gsk_krige on the same samples with the same n explicit point targets at the same k.
Median of --reps runs after one warm-up run of every shape. The device name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import gskrige  # noqa: E402

WORKLOADS = ("C2", "C3a", "C5", "C4")


def _device():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power = [s.strip() for s in q.split(",")]
    return dict(device=torch.cuda.get_device_name(0), smi_name=name, power_limit=power)


def _spec(name):
    s = gskrige.synth.config_spec(name, support="point")
    return gskrige.ProblemSpec(coords=s.coords, values=s.values, points=s.coords, **s.params)


def _timed(fn, ctx, reps):
    fn()
    walls, devs, plans = [], [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        walls.append(1e3 * (time.perf_counter() - t0))
        t = ctx.timing()
        devs.append(t["ms_plan"] + t["ms_total"])
        plans.append(t["ms_plan"])
    return statistics.median(walls), statistics.median(devs), statistics.median(plans)


def _compaction_ms(ctx, spec):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.krige_loo(spec)
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if "loo_compact" in e.key)
    return us / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = gskrige.Context(0)
    res = dict(_device())
    for name in WORKLOADS:
        spec = _spec(name)
        n, k = spec.n_samples, spec.params["max_neighbors"]
        r = dict(n=n, k=k)
        r["loo_wall_ms"], r["loo_device_ms"], r["loo_plan_ms"] = _timed(lambda: ctx.krige_loo(spec), ctx, args.reps)
        r["samples_per_s"] = n / (r["loo_wall_ms"] / 1e3)
        r["krige_wall_ms"], r["krige_device_ms"], r["krige_plan_ms"] = _timed(lambda: ctx.krige(spec), ctx, args.reps)
        ctx.set_phase_timing(True)
        ctx.krige_loo(spec)
        t = ctx.timing()
        ctx.krige(spec)
        tk = ctx.timing()
        ctx.set_phase_timing(False)
        if k > 0:
            r["loo_search_and_removal_ms"], r["loo_solve_ms"] = t["ms_search"], t["ms_solve"]
            r["loo_removal_ms"] = _compaction_ms(ctx, spec)
            r["krige_search_ms"], r["krige_solve_ms"] = tk["ms_search"], tk["ms_solve"]
            r["loo_over_krige_device"] = r["loo_device_ms"] / r["krige_device_ms"]
        else:
            r["plan_ms"], r["dubrule_pass_ms"] = t["ms_plan"], t["ms_solve"]
            r["krige_execute_ms"] = tk["ms_total"]
        res[name] = r
        print(name, json.dumps(r), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
