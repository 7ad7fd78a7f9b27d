"""Timing of gsk_krige_columns against the values-only re-solve loop it replaces; prints one JSON line.

    python scripts/columns_time.py [--reps 5] [--out FILE]

Workloads (FFTGS-like conditioning: the same data locations every time, new values per realisation):
  * local:  Ordinary Kriging, spherical, k = 32, 20 000 samples, 1448 × 1448 ≈ 2.1M grid targets at point support;
  * global: Ordinary Kriging, spherical, n = 4 000 samples, 256 × 256 = 65 536 grid targets at point support.
For m in {1, 4, 16, 64} value columns:
  * columns: one ctx.krige_columns(spec, Z) call — plan, search and factorisations once, the m means copied to host
    (pageable numpy arrays) — host clock around the call, which ends in a device synchronise;
  * loop: what a caller does today after one gsk_plan: m × (gsk_update_values + gsk_execute) into device buffers,
    then one synchronise (the plan itself and no host copy are counted, which favours the loop).
Medians of --reps runs after one warm-up of every shape. break_even_m is the smallest m of the list at which one
columns call is faster than the loop. The device name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import gskrige  # noqa: E402

MS = (1, 4, 16, 64)


def _device():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [s.strip() for s in q.split(",")]
    return dict(device=torch.cuda.get_device_name(0), smi_name=name, power_limit=power, max_sm_clock=clock)


def _spec(kind):
    if kind == "local":
        grid, n, k = (1448, 1448), 20_000, 32
    else:
        grid, n, k = (256, 256), 4_000, 0
    coords, vals = gskrige.synth.make_samples(2024, n, grid, seed_extra=k)
    return gskrige.ProblemSpec(coords=coords, values=vals, grid_dims=grid, vario_kind=gskrige.VARIO_SPHERICAL,
                               vario_range=grid[0] / 8, vario_sill=1.0, estimator=gskrige.EST_ORDINARY, max_neighbors=k)


def _median_ms(fn, reps):
    fn()
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append(1e3 * (time.perf_counter() - t0))
    return statistics.median(out)


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = gskrige.Context(0)
    res = dict(_device())
    for kind in ("local", "global"):
        spec = _spec(kind)
        n, count = spec.n_samples, spec.n_targets
        Zall = np.random.default_rng(7).normal(size=(n, max(MS)))
        d_mean = torch.empty(count, dtype=torch.float64, device="cuda")
        d_var = torch.empty(count, dtype=torch.float64, device="cuda")
        rows = {}
        for m in MS:
            Z = np.ascontiguousarray(Zall[:, :m])
            cols_ms = _median_ms(lambda: ctx.krige_columns(spec, Z), args.reps)

            def loop():
                for j in range(m):
                    ctx.update_values(Z[:, j])
                    ctx.execute(0, count, d_mean.data_ptr(), d_var.data_ptr())
                ctx.synchronize()

            ctx.plan(spec)
            loop_ms = _median_ms(loop, args.reps)
            rows[m] = dict(columns_ms=cols_ms, loop_ms=loop_ms, speedup=loop_ms / cols_ms)
            print(kind, m, json.dumps(rows[m]), file=sys.stderr, flush=True)
        be = [m for m in MS if rows[m]["columns_ms"] < rows[m]["loop_ms"]]
        res[kind] = dict(n_samples=n, targets=count, k=spec.params["max_neighbors"], by_m=rows,
                         break_even_m=be[0] if be else None)
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
