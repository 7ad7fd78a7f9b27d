#!/usr/bin/env python
"""bench.py — kriged target locations per second (mean + variance), BASELINE.json's metric.

    python bench.py --gpus N --steps K --warmup W [--config C5] [--impl reference] [--dump-outputs DIR]

The headline workload is BASELINE.json's multi-GPU configuration, **C5** (local Ordinary Kriging,
Spherical variogram, maxneighbors = 64, 1e6 3-D samples onto the 512^3 grid), at every N with **strong
scaling**: the grid is fixed, rank r of N owns the contiguous slab [T*r/N, T*(r+1)/N) of its linear index
range, every rank keeps all samples (32 MB) resident, and for N > 1 the result gather is fused into the
solve kernel (stores into every rank's symmetric-memory buffer over NVLink; NCCL all-gather with
`--gather nccl`). A "step" is one pass of the Kriging hot path (neighbour search + assemble / factor /
solve + mean and variance) over the rank's slab.

`value` is timed on the device (CUDA events on the stream the kernels run on, max over ranks) with the
samples and bins already resident in HBM; `e2e` is the same metric through the C-ABI call a host binding
makes (`gsk_krige`: host buffers in, host buffers out - upload of the samples, bin build, kernels and the
device-to-host copies of both fields inside the timed region, max over ranks).

The other BASELINE configurations (C2, C3a, C3b and a 262 144-target batch of C4, whose per-target cost is
O(n^2)) are measured in the same run, sharded over the same N ranks, with fewer steps, and reported in the
`configs` block of the same JSON line - each with its own device-resident value, e2e value and roofline
fraction. `--config X` makes X the headline instead (and `--no-secondary` skips the block).

The CPU oracle is used only for the `cpu_baseline` / `--impl reference` legs.

`--dump-outputs DIR` writes what the headline's last timed step computed, as a caller of that path receives it (the
whole job; on N > 1 the gathered job), to DIR/target.npy (linear grid index of each value), DIR/mean.npy and
DIR/variance.npy, all float64. A job larger than DUMP_BYTES is represented by a fixed, seeded sample of DUMP_SAMPLE
targets. The inputs are synthetic and seeded, so two builds run with the same arguments can be compared value for value.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for p in (ROOT, ROOT / "oracle"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import numpy as np  # noqa: E402

METRIC = "kriged locations/sec (mean+variance)"
UNIT = "locations/s"
HEADLINE = "C5"
ALL_CONFIGS = ["C1", "C2", "C3a", "C3b", "C4", "C5"]
SECONDARY = ["C2", "C3a", "C3b", "C4"]
C4_BATCH = 262_144          # targets of C4 computed per step (the full 2048^2 grid is 16 such batches)
DUMP_BYTES = 64 << 20       # --dump-outputs: at most this much in all (three float64 arrays)
DUMP_SAMPLE = 1 << 20       # targets written for a job larger than that
DUMP_SEED = 0


def host_cores() -> int:
    """Cores this process may use (torch.distributed.run exports OMP_NUM_THREADS=1: never trust that variable)."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def job_range(name, spec):
    """(first, count) of the targets one step of config `name` covers over ALL ranks."""
    T = spec.n_targets
    if name != "C4" or T <= C4_BATCH:
        return 0, T
    row = spec.grid_dims[0]
    first = (T - C4_BATCH) // 2 // row * row
    return first, C4_BATCH


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return d.get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(device)], stdout=self.tmp, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.tmp.flush()
        rows = [r.split(",") for r in Path(self.tmp.name).read_text().strip().splitlines() if r.count(",") >= 8]
        os.unlink(self.tmp.name)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except ValueError:
                continue
            for nme, val in zip(names, r[5:9]):
                if val.strip().lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # "under load" = the samples drawing more than half of the largest power seen
        load = [s for s, w in zip(sm, pw) if w >= 0.5 * max(pw)] or sm
        return {"sm_mhz": statistics.median(load), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "samples_under_load": len(load), "power_w_max": max(pw)}


def workload_name(cfg, spec, job=None):
    p = spec.params
    est = {0: "SimpleKriging", 1: "OrdinaryKriging", 2: f"UniversalKriging(degree={p['uk_degree']})"}[p["estimator"]]
    vg = {0: "Gaussian", 1: "Spherical", 2: "Exponential"}[p["vario_kind"]]
    k = p["max_neighbors"]
    grid = "x".join(str(g) for g in spec.grid_dims)
    s = (f"{cfg}: {'local' if k else 'global'} {est} {vg}Variogram(range={p['vario_range']:g})"
         f"{f' maxneighbors={k}' if k else ''}, {spec.n_samples} {spec.dim}D samples -> {grid} grid, "
         f"block support q={spec.support[0].shape[0]}")
    if job is not None and job[1] != spec.n_targets:
        s += f"; {job[1]} consecutive targets per step (of {spec.n_targets})"
    return s


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU path on the box's host cores
# ------------------------------------------------------------------------------------------------
def oracle_rate(O, spec, first_mid, sample, nthreads, passes):
    sl = spec.with_slab(first_mid - sample // 2, sample)
    best = 1e30
    for _ in range(passes):
        c0 = time.perf_counter(); O.krige(sl, nthreads=nthreads); best = min(best, time.perf_counter() - c0)
    return sample / best, best


def calibrated_sample(O, spec, job, cores, seconds):
    """A bounded sample of the job's targets (consecutive, from the middle of the job) sized so that one oracle
    pass over it takes about `seconds` on `cores` threads. The first (small) pass also builds the searcher."""
    jf, jc = job
    mid = jf + jc // 2
    probe = min(jc, 16_384)
    O.krige(spec.with_slab(mid - probe // 2, probe), nthreads=cores)          # builds + caches the KD-tree
    rate, _ = oracle_rate(O, spec, mid, probe, cores, 2)
    sample = int(min(jc, max(probe, rate * seconds)))
    sample = max(1024, sample // 1024 * 1024)
    return min(sample, jc), mid


def run_reference(args):
    """--impl reference: the reference's CPU path. The reference is pure Julia and no julia binary exists in this
    image, so this times the oracle port (oracle/gsk_oracle.c: KD-tree search, per-target LU, OpenMP over targets on
    ALL host cores - the thread count is passed explicitly) on the same config/metric. Each step is a bounded sample
    of the workload. Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import gskrige
    import oracle_py as O
    name = args.config
    spec = gskrige.synth.config_spec(name)
    job = job_range(name, spec)
    cores = host_cores()
    if spec.params["max_neighbors"] == 0 and spec.n_samples > 2000:
        # C4: one O(n^3) LU on the CPU is minutes; time the test-sized global config instead and say so
        line = {"impl": "reference", "unavailable": f"{name}: the CPU port needs a {spec.n_samples + 1}^2 LU per call; use --config C5/C2/C3a/C3b/C1"}
        print(json.dumps(line), flush=True)
        return
    # every step ~ (200 s / (K + W)) of CPU time, at most 6 s, so that the whole run ends within a few minutes
    per_step = max(0.5, min(6.0, 200.0 / max(1, args.steps + args.warmup)))
    sample, mid = calibrated_sample(O, spec, job, cores, per_step) if args.cpu_sample <= 0 else (min(args.cpu_sample, job[1]), job[0] + job[1] // 2)
    slab = spec.with_slab(mid - sample // 2, sample)
    for _ in range(args.warmup):
        O.krige(slab, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        O.krige(slab, nthreads=cores)
    dt = (time.perf_counter() - t0) / max(1, args.steps)
    value = sample / dt
    s1 = max(1024, sample // 16)
    v1, _ = oracle_rate(O, spec, mid, s1, 1, 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(name, spec, job), "sample_targets": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample} consecutive targets from the middle of the {name} grid per step (KD-tree built once, "
                                   f"as preprocess does; per-target search + LU + solve, OpenMP, {cores} threads passed explicitly)",
                         "value_1_thread": v1, "sample_1_thread": f"{s1} targets, 1 thread (the reference's own loop is serial)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference is pure Julia (no julia binary in this image); timed: the C oracle port on all host cores",
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# product arm
# ------------------------------------------------------------------------------------------------
class Env:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import gskrige
        self.torch, self.dist, self.gsk, self.args = torch, dist, gskrige, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a B200: the Kriging path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.cpu_group = None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
            self.cpu_group = dist.new_group(backend="gloo")   # host-only barrier: an NCCL barrier keeps a kernel spinning on the waiting GPUs
        self.stream = torch.cuda.current_stream()
        self.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=self.dev)   # 256 MB > 126 MB L2
        self.peaks = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


class Workload:
    """One BASELINE config planned on this rank's GPU, its slab, its output buffers and its step()."""

    def __init__(self, env: Env, name: str):
        gsk, torch, dist = env.gsk, env.torch, env.dist
        self.env, self.name = env, name
        self.spec = spec = gsk.synth.config_spec(name)
        self.job = job_range(name, spec)
        jf, jc = self.job
        if env.args.targets:
            jc = min(jc, env.args.targets * env.world)
            self.job = (jf, jc)
        first, count = gsk.slab_bounds(jc, env.rank, env.world)
        self.first, self.count = jf + first, count
        self.k = spec.params["max_neighbors"]
        self.ctx = gsk.Context(env.local_rank)
        self.ctx.set_stream(env.stream.cuda_stream)
        self.ctx.plan(spec)                                   # samples + bins (or the global factor) resident in HBM
        self.plan_ms = self.ctx.timing()["ms_plan"]
        self.d_mean = torch.empty(count, dtype=torch.float64, device=env.dev)
        self.d_var = torch.empty(count, dtype=torch.float64, device=env.dev)
        self.hdl = None
        self.gather_mode = "single GPU"
        equal = count * env.world == jc
        if env.world > 1:
            if env.args.gather != "nccl" and equal:
                try:
                    import torch.distributed._symmetric_memory as symm_mem
                    self.sbuf = symm_mem.empty(2 * jc, dtype=torch.float64, device=env.dev)
                    self.hdl = symm_mem.rendezvous(self.sbuf, dist.group.WORLD)
                    ptrs = [int(p) for p in self.hdl.buffer_ptrs]
                    self.mean_ptrs, self.var_ptrs, self.use_mc = ptrs, [p + 8 * jc for p in ptrs], False
                    if env.args.gather == "multicast":
                        mc = int(getattr(self.hdl, "multicast_ptr", 0) or 0)
                        if mc:
                            self.mean_ptrs, self.var_ptrs, self.use_mc = [mc], [mc + 8 * jc], True
                    self.gather_mode = ("results stored by the compute kernels into every rank's symmetric-memory buffer over NVLink "
                                        + ("(one NVLS multicast store per value)" if self.use_mc else "(P2P stores to each peer)")
                                        + ", device-side barrier per step")
                except Exception as exc:  # noqa: BLE001 - fall back to NCCL, say so in the JSON line
                    self.hdl = None
                    self.gather_mode = f"NCCL all-gather (symmetric memory unavailable: {type(exc).__name__})"
            if self.hdl is None:
                self.g_mean = torch.empty(jc, dtype=torch.float64, device=env.dev)
                self.g_var = torch.empty(jc, dtype=torch.float64, device=env.dev)
                if env.args.gather == "nccl" or not equal:
                    self.gather_mode = "NCCL all-gather of mean and variance inside the timed step"

    def step(self):
        env = self.env
        if self.hdl is not None:
            self.ctx.execute_peers(self.first, self.count, self.mean_ptrs, self.var_ptrs,
                                   out_offset=env.rank * self.count, multicast=self.use_mc)
            self.hdl.barrier(channel=0)                   # every rank's stores have landed everywhere
            return
        self.ctx.execute(self.first, self.count, self.d_mean.data_ptr(), self.d_var.data_ptr())
        if env.world > 1:                                 # result gather: NCCL all-gather over NVLink
            from gskrige.sharding import gather_slabs
            if self.count * env.world == self.job[1]:
                env.dist.all_gather_into_tensor(self.g_mean, self.d_mean)
                env.dist.all_gather_into_tensor(self.g_var, self.d_var)
            else:
                self.g_mean = gather_slabs(self.d_mean, self.job[1])
                self.g_var = gather_slabs(self.d_var, self.job[1])

    def timed_steps(self, steps, sampler_rank0=False):
        """K steps, each bracketed by CUDA events on the launching stream, L2 flushed between; returns
        (ms_per_step as max over ranks of the summed device time / K, wall seconds, clocks or None)."""
        env, torch = self.env, self.env.torch
        sampler = ClockSampler(env.local_rank) if (sampler_rank0 and env.rank == 0) else None
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        try:
            env.barrier()
            wall0 = time.perf_counter()
            for a, b in evs:
                env.flush.zero_()
                a.record(env.stream)
                self.step()
                b.record(env.stream)
            env.barrier()
            wall = time.perf_counter() - wall0
        finally:                                          # a failing step must not leave nvidia-smi polling
            clocks = sampler.stop() if sampler else None
        dev_ms = env.max_over_ranks(sum(a.elapsed_time(b) for a, b in evs))
        return dev_ms / steps, wall, clocks

    def dump_outputs(self, out_dir):
        """mean and variance of the job as the last step left them (see --dump-outputs), on the rank that calls it"""
        torch, (jf, jc) = self.env.torch, self.job
        if self.hdl is not None:
            mean, var = self.sbuf[:jc], self.sbuf[jc:]
        elif self.env.world > 1:
            mean, var = self.g_mean, self.g_var
        else:
            mean, var = self.d_mean, self.d_var
        if 3 * 8 * jc <= DUMP_BYTES:
            pick = np.arange(jc, dtype=np.int64)
        else:
            pick = np.sort(np.random.default_rng(DUMP_SEED).choice(jc, DUMP_SAMPLE, replace=False))
        sel = torch.from_numpy(pick).to(self.env.dev)
        out = Path(out_dir)
        out.mkdir(parents=True, exist_ok=True)
        np.save(out / "target.npy", (jf + pick).astype(np.float64))
        np.save(out / "mean.npy", mean.index_select(0, sel).cpu().numpy())
        np.save(out / "variance.npy", var.index_select(0, sel).cpu().numpy())

    def check_gather(self):
        """the gathered field must be identical on every rank and hold this rank's slab at its place"""
        env, torch, dist = self.env, self.env.torch, self.env.dist
        if self.hdl is None:
            return
        self.ctx.execute(self.first, self.count, self.d_mean.data_ptr(), self.d_var.data_ptr())
        torch.cuda.synchronize()
        jc = self.job[1]
        full_mean = self.sbuf[:jc]
        own = full_mean[env.rank * self.count:(env.rank + 1) * self.count]
        assert torch.equal(torch.nan_to_num(own, nan=-7.0), torch.nan_to_num(self.d_mean, nan=-7.0)), "fused gather: own slab differs"
        chk = torch.stack([torch.nan_to_num(full_mean).sum(), torch.nan_to_num(self.sbuf[jc:]).sum()])
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        assert torch.equal(lo, hi), "fused gather: ranks hold different gathered fields"

    def phases(self, n):
        """search / solve kernel times with events around each launch (extra steps, not part of `value`)"""
        ps, pv, launches = [], [], 0
        self.ctx.set_phase_timing(True)
        for _ in range(n):
            self.env.flush.zero_()
            self.ctx.execute(self.first, self.count, self.d_mean.data_ptr(), self.d_var.data_ptr())
            tt = self.ctx.timing()
            ps.append(tt["ms_search"]); pv.append(tt["ms_solve"]); launches = int(tt["launches"])
        self.ctx.set_phase_timing(False)
        self.env.torch.cuda.synchronize()
        return statistics.median(ps), statistics.median(pv), launches

    def e2e(self, warm, steps):
        """the C-ABI call with host buffers (pinned): H2D + plan + kernels + D2H inside the timed region"""
        env, torch, gsk = self.env, self.env.torch, self.env.gsk
        h_mean = torch.empty(self.count, dtype=torch.float64).pin_memory().numpy()
        h_var = torch.empty(self.count, dtype=torch.float64).pin_memory().numpy()
        slab = self.spec.with_slab(self.first, self.count)
        ectx = gsk.Context(env.local_rank)
        for _ in range(warm):
            ectx.krige_into(slab, h_mean, h_var)
        env.barrier()
        e0 = time.perf_counter()
        for _ in range(steps):
            ectx.krige_into(slab, h_mean, h_var)
        env.barrier()
        e2e_s = env.max_over_ranks((time.perf_counter() - e0) / steps)
        self.ctx.execute(self.first, self.count, self.d_mean.data_ptr(), self.d_var.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(h_mean, self.d_mean.cpu().numpy(), equal_nan=True), "e2e and resident paths disagree"
        ectx.close()
        del h_mean, h_var
        spec = self.spec
        h2d = spec.n_samples * (spec.dim + 1) * 8 + 3 * spec.support[0].shape[0] * 8
        return {"value": self.job[1] / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 16 * self.count,
                "ms_per_step": e2e_s * 1e3, "steps": steps,
                "api": "gsk_krige (C ABI, pinned host buffers; sample upload + bin build / factorisation + kernels + D2H per call)"}

    def launches_per_chunk(self):
        """Kernels per chunk of <= 2^20 targets on the local path: the compact-key search, its exact redo pass (both
        launched whenever the sample index fits the key: n <= 2^24 and no ball) and the solve kernel."""
        p = self.spec.params
        ball = p["ball_radius"] == p["ball_radius"]
        return 3 if (self.spec.n_samples <= (1 << 24) and not ball) else 2

    def roofline(self, ms_per_step, solve_ms, search_ms, launches, dfma, dmma):
        gsk, spec, k = self.env.gsk, self.spec, self.k
        flops_t = gsk.synth.algorithmic_flops_per_target(spec)
        hbm_peak, how = peaks()
        traffic = None
        tf = ROOT / "profiles" / "roofline_traffic.json"
        if tf.exists():
            per_target = json.loads(tf.read_text()).get("bytes_per_target", {}).get(self.name)
            if per_target is not None and k:
                traffic = per_target * self.count / max(1, launches // self.launches_per_chunk())   # per launch, like `achieved`'s launch set / its launches
        extra = {}
        count = self.count
        if k:
            solve_ms = solve_ms or ms_per_step
            achieved = flops_t * count / (solve_ms * 1e-3) / 1e12          # all solve launches of a step together
            kernel = "local_solve_small_kernel" if (k <= 20 and spec.params["estimator"] != 2) else "local_solve_kernel"
            bound, peak, frac = "fp64", dfma, achieved / dfma
            step_ms = (search_ms + solve_ms) if search_ms else ms_per_step
            extra = {"frac_step": flops_t * count / (step_ms * 1e-3) / 1e12 / dfma,
                     "frac_step_note": "same algorithmic flops over search + solve kernel time (the whole per-target path)"}
            nlaunch = max(1, launches // self.launches_per_chunk())
        else:
            # global path: the Gram formulation needs only the forward triangular solve, i.e. n^2 flop per target
            # instead of the canonical 2(n+c)^2 - both are reported; frac uses the EXECUTED flops (conservative)
            solve_ms = ms_per_step
            achieved = flops_t * count / (ms_per_step * 1e-3) / 1e12
            np_ = -(-spec.n_samples // 128) * 128
            executed = float(np_) * np_ * count / (ms_per_step * 1e-3) / 1e12
            kernel, bound, peak, frac = "ygemm_dmma_kernel (+rhs_kernel, epilogue)", "tensor", dmma, executed / dmma
            extra = {"achieved_executed": executed, "frac_canonical": achieved / dmma,
                     "note": "tensor = FP64 mma.sync (DMMA); tcgen05 has no FP64 kind. frac = executed flops / measured DMMA peak"}
            nlaunch = 1
        return {"bound": bound, "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": frac,
                "traffic": traffic, **extra,
                "peak_source": "measured in this run (gsk_measure_fp64_peak): DFMA loop %.1f TFLOP/s, DMMA m16n8k16 loop %.1f TFLOP/s" % (dfma, dmma),
                "algorithmic_flops_per_target": flops_t, "targets_per_launch_set": count, "kernel_ms_per_step": solve_ms,
                "launches_per_step": nlaunch,
                "hbm": {"achieved_gbs": 16.0 * count / (solve_ms * 1e-3) / 1e9, "peak_gbs": hbm_peak, "peak_source": how,
                        "algorithmic_bytes_per_target": 16}}

    def close(self):
        self.ctx.close()
        for a in ("d_mean", "d_var", "g_mean", "g_var", "sbuf", "hdl"):
            if hasattr(self, a):
                setattr(self, a, None)
        self.env.torch.cuda.empty_cache()


def measure_secondary(env: Env, name: str, dfma, dmma):
    """A non-headline BASELINE config in the same run: fewer steps, same rules (warm-up >= 3, L2 flushed, device events,
    max over ranks)."""
    w = Workload(env, name)
    for _ in range(3):
        w.step()
    env.barrier()
    probe_ms, _, _ = w.timed_steps(1)
    steps = int(max(3, min(20, 2500.0 / max(probe_ms, 1e-3))))
    ms, wall, _ = w.timed_steps(steps)
    search_ms, solve_ms, launches = w.phases(3 if probe_ms < 1000 else 1)
    e2e = w.e2e(1, 3 if probe_ms < 1000 else 2)
    rf = w.roofline(ms, solve_ms, search_ms, launches, dfma, dmma)
    out = {"workload": workload_name(name, w.spec, w.job), "value": w.job[1] / (ms * 1e-3), "ms_per_step": ms, "steps": steps,
           "warmup": 4, "targets_per_gpu": w.count, "e2e": {k: e2e[k] for k in ("value", "ms_per_step", "h2d_bytes_per_step", "d2h_bytes_per_step")},
           "frac": rf["frac"], "frac_step": rf.get("frac_step"), "bound": rf["bound"], "kernel": rf["kernel"],
           "kernel_ms": rf["kernel_ms_per_step"], "phases_ms": {"plan": w.plan_ms, "search": search_ms, "solve": solve_ms},
           "algorithmic_flops_per_target": rf["algorithmic_flops_per_target"]}
    if "achieved_executed" in rf:
        out["frac_canonical"] = rf["frac_canonical"]
    w.close()
    return out


def measure_callers(env: Env):
    """SURVEY §8f rows that sit on the same kernels, through the public API with host buffers (documentation figures,
    a few seconds in total): the IDW / LWR solvers on the C2 shape, and sequential Gaussian simulation (plan = masked
    search + weights for the whole path; realisations = level-scheduled recurrence)."""
    gsk, torch = env.gsk, env.torch
    out = {}
    ctx = gsk.Context(env.local_rank)
    try:
        base = gsk.synth.config_spec("C2")
        T = int(np.prod(base.grid_dims))
        for nm, sv in (("idw", gsk.SOLVER_IDW), ("lwr", gsk.SOLVER_LWR)):
            spec = gsk.ProblemSpec(coords=base.coords, values=base.values, grid_dims=base.grid_dims, solver=sv, idw_exponent=2.0,
                                   max_neighbors=20)
            ctx.krige(spec)
            t0 = time.perf_counter()
            for _ in range(3):
                ctx.krige(spec)
            dt = (time.perf_counter() - t0) / 3
            out[nm] = {"workload": f"{nm.upper()} solver, C2 shape (1000x1000 grid, 10 000 samples, maxneighbors=20)",
                       "value": T / dt, "unit": UNIT, "ms_per_call": dt * 1e3, "api": "gsk_krige, host buffers"}
        # SGS: 512x512 grid, 100 data, spherical variogram, maxneighbors = 10, random path
        dims, k, nreal = (512, 512), 10, 64
        n = dims[0] * dims[1]
        rng = np.random.default_rng(0)
        gx, gy = np.meshgrid(np.arange(dims[0]) + 0.5, np.arange(dims[1]) + 0.5)
        cs = [gx.ravel().copy(), gy.ravel().copy()]
        data = rng.choice(n, 100, replace=False)
        order = rng.permutation(n)
        isdata = np.zeros(n, dtype=bool)
        isdata[data] = True
        visit = order[~isdata[order]]
        rank = np.full(n, -1, dtype=np.int64)
        rank[visit] = np.arange(len(visit))
        vals = np.where(isdata, rng.standard_normal(n), 0.0)
        kw = dict(vario_kind=gsk.VARIO_SPHERICAL, vario_range=20.0, max_neighbors=k)
        ctx.sgs_plan(cs, rank, **kw)
        t0 = time.perf_counter()
        ctx.sgs_plan(cs, rank, **kw)
        t_plan = time.perf_counter() - t0
        z = rng.standard_normal((nreal, n))
        ctx.sgs_sample(z[:1], values=vals)
        t0 = time.perf_counter()
        res = ctx.sgs_sample(z, values=vals)
        t_abi = time.perf_counter() - t0
        tk = ctx.timing()
        dz, dv = torch.from_numpy(z).to(env.dev), torch.from_numpy(vals).to(env.dev)
        dout = torch.empty_like(dz)
        torch.cuda.synchronize(env.dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.set_stream(env.stream.cuda_stream)
        ctx.sgs_sample_device(nreal, dv.data_ptr(), dz.data_ptr(), dout.data_ptr())
        e0.record(env.stream)
        ctx.sgs_sample_device(nreal, dv.data_ptr(), dz.data_ptr(), dout.data_ptr())
        e1.record(env.stream)
        torch.cuda.synchronize(env.dev)
        ms_dev = e0.elapsed_time(e1)
        same = bool(np.array_equal(dout.cpu().numpy(), res))
        out["sgs"] = {"workload": f"SGS, {dims[0]}x{dims[1]} grid, 100 data, spherical variogram, maxneighbors={k}, random path, {nreal} realisations",
                      "plan_ms": t_plan * 1e3, "value": nreal * n / t_abi, "unit": "simulated locations/s",
                      "ms_per_call": t_abi * 1e3, "api": "gsk_sgs_sample, pageable host buffers (draws in, realisations out)",
                      "device_resident": {"value": nreal * n / (ms_dev * 1e-3), "ms_per_call": ms_dev, "launches": int(tk["launches"]),
                                          "api": "gsk_sgs_sample_device", "same_bytes_as_host_call": same}}
    except Exception as exc:  # noqa: BLE001 - informational block
        out["error"] = f"{type(exc).__name__}: {exc}"
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of the headline config")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=HEADLINE, choices=ALL_CONFIGS)
    ap.add_argument("--cpu-sample", type=int, default=0, help="targets per step of the CPU legs (0: calibrated to a few seconds)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the `configs` block (other BASELINE configs)")
    ap.add_argument("--targets", type=int, default=0, help="limit the per-rank slab (debug)")
    ap.add_argument("--gather", default="multicast", choices=["peer", "multicast", "nccl"],
                    help="N>1 result gather: stores into every rank's symmetric-memory buffer fused in the solve kernel "
                         "(peer), the same through one NVLS multicast store (multicast), or an NCCL all-gather (nccl)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline's last timed step (target index, mean, variance) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the product path's outputs; the reference arm times a calibrated CPU sample")
    if args.impl == "reference":
        run_reference(args)
        return

    env = Env(args)
    torch, dist = env.torch, env.dist
    name = args.config
    w = Workload(env, name)
    warm = max(args.warmup, 3)
    for _ in range(warm):
        w.step()
    env.barrier()
    launches_per_step = int(w.ctx.timing()["launches"])

    ms_per_step, wall, clocks = w.timed_steps(args.steps, sampler_rank0=True)
    value = w.job[1] / (ms_per_step * 1e-3)
    if args.dump_outputs and env.rank == 0:              # before any later leg overwrites the step's buffers
        w.dump_outputs(args.dump_outputs)
    w.check_gather()

    long_step = ms_per_step > 1000.0
    search_ms, solve_ms, launches = w.phases(1 if long_step else min(args.steps, 10))
    dfma, dmma = w.ctx.measure_fp64_peak()
    e2e = w.e2e(1 if long_step else 2, 2 if long_step else max(3, min(args.steps, 10)))
    roof = w.roofline(ms_per_step, solve_ms, search_ms, launches, dfma, dmma)
    spec, job, count, plan_ms, gather_mode = w.spec, w.job, w.count, w.plan_ms, w.gather_mode
    w.close()

    # N > 1, additionally: the whole job through ONE call of the single-process multi-GPU entry point (gsk_krige_multi —
    # what a Julia host driving all GPUs of the box from one process uses): rank 0 calls it over all N devices while the
    # other ranks idle at the barrier. Host buffers are page-locked; sample upload, bin build, kernels and the copies
    # back are inside the timed region.
    if env.world > 1:
        if env.rank == 0:
            try:
                hm = torch.empty(job[1], dtype=torch.float64).pin_memory().numpy()
                hv = torch.empty(job[1], dtype=torch.float64).pin_memory().numpy()
                whole = spec.with_slab(job[0], job[1])
                env.gsk.krige_multi(whole, list(range(env.world)), out=(hm, hv))      # warm: contexts, buffers
                reps = 1 if long_step else 3
                m0 = time.perf_counter()
                for _ in range(reps):
                    env.gsk.krige_multi(whole, list(range(env.world)), out=(hm, hv))
                ms = (time.perf_counter() - m0) / reps * 1e3
                e2e["single_process"] = {"value": job[1] / (ms * 1e-3), "ms_per_step": ms, "steps": reps,
                                         "api": "gsk_krige_multi (one process, one host thread and context per GPU, page-locked host buffers)"}
                del hm, hv
            except Exception as exc:  # noqa: BLE001 - informational leg
                e2e["single_process"] = {"error": f"{type(exc).__name__}: {exc}"}
        # the other ranks wait on the HOST (gloo): a waiting NCCL barrier is a spinning kernel on their GPUs, and a GPU
        # time-slices between the processes that use it — rank 0's worker for that device would run at half speed
        dist.barrier(group=env.cpu_group)
        env.barrier()

    configs = {}
    if not args.no_secondary and not args.targets:
        for other in SECONDARY + [HEADLINE]:
            if other == name:
                continue
            try:
                configs[other] = measure_secondary(env, other, dfma, dmma)
            except Exception as exc:  # noqa: BLE001 - a failing secondary config must not hide the headline line
                configs[other] = {"error": f"{type(exc).__name__}: {exc}"}
            env.barrier()

    callers = {}
    if not args.no_secondary and not args.targets:
        if env.rank == 0:
            callers = measure_callers(env)
        env.barrier()

    if env.rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": env.world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(name, spec, job), "targets_per_step": job[1], "targets_per_gpu": count,
                       "l2": "flushed between timed steps (256 MB write)",
                       "multi_gpu": ("strong scaling: the fixed grid is cut into contiguous slabs of its linear index range, one per rank, "
                                     "samples replicated; " + gather_mode) if env.world > 1 else "single GPU"},
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": int(launches_per_step * args.steps),
            "roofline": roof,
            "phases_ms": {"plan": plan_ms, "search": search_ms, "solve": solve_ms},
            "wall_s_timed_region": wall,
            "configs": configs,
            "callers": callers,
        }
        if not args.no_cpu_baseline and env.world == 1:
            import oracle_py as O
            cores = host_cores()
            if spec.params["max_neighbors"] == 0 and spec.n_samples > 2000:
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": cores, "kind": "port",
                                        "sample": "not run: one (n+1)^2 LU + O(n^2) per target on the CPU"}
            else:
                sample, mid = calibrated_sample(O, spec, job, cores, 4.0) if args.cpu_sample <= 0 else (min(args.cpu_sample, job[1]), job[0] + job[1] // 2)
                v, best = oracle_rate(O, spec, mid, sample, cores, 3)
                # the reference's own loop is serial (krig.jl:180,205 use no threads): the 1-thread figure is its analogue
                s1 = max(1024, sample // 16)
                v1, _ = oracle_rate(O, spec, mid, s1, 1, 1)
                line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                        "sample": f"{sample} consecutive targets from the middle of the grid, best of 3 passes of {best:.2f} s "
                                                  f"(C oracle port: KD-tree built once as preprocess does, per-target search + LU + solve, OpenMP, {cores} threads)",
                                        "value_1_thread": v1, "sample_1_thread": f"{s1} consecutive targets, 1 thread"}
        print(json.dumps(line), flush=True)
    if env.world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
