#!/usr/bin/env python
"""Benchmarks of the FiniteBLR inference path (BASELINE.json), one JSON line per run (rank 0).

    python bench.py --gpus N --steps K --warmup W                  # headline: cfg3, our arm (libblr_cuda on B200)
    python bench.py --config cfg2|cfg3|cfg4|cfg5 ...               # the other BASELINE configs, same one-line contract
    python bench.py --impl reference [--config ...] ...            # the reference's CPU op sequence on the box's host cores
    python bench.py ... --dump-outputs DIR                         # also write the last timed step's results as DIR/<name>.npy

Configs (BASELINE.json `configs`):
  cfg3  diagonal-noise BLR posterior+logpdf, N = 2^24, D = 1024, ColVecs, N-sharded (the config `metric` is quoted on; default)
  cfg2  the same at N = 2^20, D = 256
  cfg5  BasisFunctionRegressor with random Fourier features (D = 4096, d_in = 32), N = 2^22, posterior+logpdf, ϕ evaluated on
        the device at every call (src/basis_function_regression.jl:41) and never leaving it
  cfg4  marginals (mean_and_var) on 2^26 test points at D = 512 (value), plus rand with S = 64 function samples (extra key);
        test points sharded, 2^24 per GPU at most (the full 256 GiB matrix needs >= 4 B200s)

A "step" is one pass of the path over the whole synthetic input (generated in place on the device with Philox; inputs are far
larger than the 126 MB L2, so no flush is needed between steps).  N is fixed as GPUs are added => strong scaling; the only
collective is ONE NCCL sum-allreduce of the packed statistics per step (none on the prediction side).  Parity: every run
checks its result -- posterior+logpdf configs against the committed log marginal likelihood of the same synthetic data set
(profiles/bench_expected.json, relative 1e-11: the value must not depend on the number of GPUs), cfg4 against torch on
sampled blocks of test points -- and exits non-zero on a mismatch.

--dump-outputs DIR (rank 0, our arm): after the timed steps, the arrays the timed path returned in its LAST step, float64,
one DIR/<name>.npy each -- posterior+logpdf configs: posterior_mean, posterior_precision, logpdf; cfg4: mean, var, rand
(device draws), rand_supplied_draws.  An array of more than 2^20 elements is stored as its values at a fixed seeded set of
flat (row-major) positions, the same for every run of the same shape, so that two builds can be compared output for
output; the inputs are generated from --seed alone.  cfg4 with several GPUs dumps rank 0's shard of the test points.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NOMINAL_FP64_TFLOPS = 37.2  # 148 SM x 64 DFMA/clk x 2 x 1.965 GHz (BASELINE.md)
EXPECTED_PATH = os.path.join(ROOT, "profiles", "bench_expected.json")
TRAFFIC_PATH = os.path.join(ROOT, "profiles", "gram_traffic.json")
DUMP_MAX_ELEMS = 1 << 20  # 8 MiB of float64 per dumped array; at most four arrays per config keep a dump under 64 MB

CONFIGS = {
    "cfg3": dict(kind="infer", n=1 << 24, dim=1024, unit="obs/s", metric="obs/s for posterior+logpdf (fp64, N=16M, D=1024)"),
    "cfg2": dict(kind="infer", n=1 << 20, dim=256, unit="obs/s", metric="obs/s for posterior+logpdf (fp64, N=1M, D=256)"),
    "cfg5": dict(kind="rff", n=1 << 22, dim=4096, din=32, unit="obs/s",
                 metric="obs/s for BasisFunctionRegressor (RFF D=4096) posterior+logpdf (fp64, N=4M)"),
    "cfg4": dict(kind="predict", n=1 << 26, dim=512, samples=64, unit="points/s",
                 metric="test points/s for marginals mean_and_var (fp64, N*=64M, D=512)"),
}


def gram_flops(N, D):  # algorithmic flops of the Gram kernel (SURVEY.md 8d): SYRK lower + r
    return float(N) * D * (D + 1) + 2.0 * N * D


def path_flops(N, D):  # whole posterior+logpdf path
    return float(N) * D * (D + 1) + 4.0 * N * D + D**3 / 3.0 + 4.0 * D * D


def resolve(args, world):
    """Workload of this run: the named config with any --n-obs / --dim override applied (overrides are for sweeps and tools;
    the JSON names what actually ran)."""
    c = dict(CONFIGS[args.config])
    if args.n_obs:
        c["n"] = args.n_obs
    if args.dim:
        c["dim"] = args.dim
    if c["kind"] == "predict":
        c["n"] = min(c["n"], world << args.max_log2_per_gpu)
    return c


def config_dict(args, c, world):
    """Identical for both arms (the driver compares it): a function of the arguments and the world size only."""
    N, D = c["n"], c["dim"]
    if c["kind"] == "infer":
        wl = f"diagonal-noise BLR posterior+logpdf, N={N}, D={D}, fp64, ColVecs, N-sharded over {world} GPU(s)"
        extra = {"prior": "mw=0, Λw=I" if args.prior_mean == "zero" else "mw~N(0, 0.01 I) (non-zero prior mean: δ = y - X'mw read from X), Λw=I",
                 "noise": "homoscedastic 0.37 I" if args.scalar_noise else "heteroscedastic diagonal exp(N(0,1))",
                 "parallelism": f"obs-sharded x{world}, one NCCL allreduce of D^2+D+3 doubles"}
    elif c["kind"] == "rff":
        wl = (f"BasisFunctionRegressor, ϕ = random Fourier features sqrt(2/D) cos(Wx+b), d_in={c['din']}, D={D}, N={N}, posterior+logpdf, "
              f"fp64, ϕ(x) evaluated on the device per call, N-sharded over {world} GPU(s)")
        extra = {"prior": "mw=0, Λw=I", "noise": "heteroscedastic diagonal exp(N(0,1))",
                 "parallelism": f"obs-sharded x{world}, one NCCL allreduce of D^2+D+3 doubles"}
    else:
        wl = (f"posterior marginals mean_and_var on N*={N} test points, D={D}, fp64, ColVecs (+ rand with S={c['samples']} function samples), "
              f"test points sharded over {world} GPU(s)")
        extra = {"posterior": "from a diagonal-noise fit on 2^20 observations, prior mw=0, Λw=I", "noise": "0.1 I at the test points",
                 "parallelism": f"test points sharded x{world}, no collective"}
    per_gpu = N / world * (c.get("din", D) if c["kind"] == "rff" else D) * 8 / 2**30
    out = {"workload": wl, "name": args.config, "n": N, "dim": D,
           "l2": "inputs (%.2f GiB per GPU%s) far larger than the 126 MB L2; no flush needed" %
                 (per_gpu, "; ϕ(x) %.1f GiB" % (N / world * D * 8 / 2**30) if c["kind"] == "rff" else "")}
    out.update(extra)
    return out


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock, power and throttle reasons of one GPU sampled DURING the timed region: NVML in-process every 5 ms (a timed
    region can be as short as ~10 ms at cfg2 -- `nvidia-smi -lms` needs longer than that just to start), nvidia-smi as the
    fallback when pynvml is unavailable."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, device: int):
        self.rows, self.proc, self.nvml, self.samples, self._stop = [], None, None, [], threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[device]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else device
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self._sample_nvml()  # fail here, not in the thread, if a query is unsupported
            self.samples.clear()
            self.t = threading.Thread(target=self._pump_nvml, daemon=True)
            self.t.start()
            return
        except Exception:  # noqa: BLE001  (no pynvml / NVML error: fall back to the CLI)
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(device), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _sample_nvml(self):
        n = self.nvml
        sm = float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
        pw = n.nvmlDeviceGetPowerUsage(self.h) / 1000.0
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        self.samples.append((sm, pw, int(get(self.h))))

    def _pump_nvml(self):
        while not self._stop.is_set():
            try:
                self._sample_nvml()
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.005)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if self.nvml is not None:
            self._stop.set()
            self.t.join(timeout=2)
            if not self.samples:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
            n = self.nvml
            masks = {"hw_slowdown": getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            seen = 0
            for _, _, m in self.samples:
                seen |= m
            return {"sm_mhz": statistics.median(x[0] for x in self.samples), "sm_max_mhz": self.mx,
                    "power_w_max": max(x[1] for x in self.samples), "samples": len(self.samples), "source": "nvml, 5 ms period",
                    "reasons": sorted(k for k, v in masks.items() if seen & v)}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1])); pw.append(float(p[2]))
            except ValueError:
                continue
            for nm, val in zip(self.NAMES, p[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "source": "nvidia-smi -lms 100", "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ host placement
def bind_to_gpu_numa(device: int):
    """Pin this process (and the page-locked buffers it allocates afterwards: first touch) to the CPUs NVML reports as local
    to the GPU.  With 8 ranks streaming from host memory at once, buffers on the wrong socket cross the inter-socket link."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus = (cpus & allowed) or allowed
        os.sched_setaffinity(0, cpus)
        node = None
        try:
            bdf = pynvml.nvmlDeviceGetPciInfo(h).busId
            bdf = (bdf.decode() if isinstance(bdf, bytes) else bdf).lower()
            node = int(open(f"/sys/bus/pci/devices/{bdf[-12:]}/numa_node").read())
        except Exception:
            pass
        return {"bound": True, "cpus": len(cpus), "numa_node": node, "restore": allowed}
    except Exception as e:  # pragma: no cover
        return {"bound": False, "why": f"{type(e).__name__}: {e}"}


def use_all_host_threads(restore=None):
    """torchrun exports OMP_NUM_THREADS=1 and the e2e leg narrows the affinity; the CPU arm is meant to use every host core."""
    if restore:
        try:
            os.sched_setaffinity(0, restore)
        except OSError:
            pass
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        from threadpoolctl import threadpool_limits

        threadpool_limits(limits=cores)
    except Exception:  # pragma: no cover
        pass
    return cores


# ------------------------------------------------------------------------------------------------ CPU reference arm
def cpu_sample(D, n_sample, seed=0):
    rng = np.random.default_rng(seed)
    X = np.asfortranarray(rng.standard_normal((D, n_sample)))
    σ2 = np.exp(rng.standard_normal(n_sample))
    y = X.T @ rng.standard_normal(D) + np.sqrt(σ2) * rng.standard_normal(n_sample)
    return X, y, σ2


def cpu_pass_factory(args, c):
    """-> (callable running ONE bounded-sample pass of the reference's own op sequence for this config, units per pass,
    description).  posterior and logpdf are two independent calls, as a user of the reference incurs (:56,:61)."""
    from oracle import blr_oracle as ref

    D = c["dim"]
    if c["kind"] == "infer":
        n = args.cpu_sample or (1 << 15 if D >= 512 else 1 << 17)
        X, y, σ2 = cpu_sample(D, n)
        f = ref.BayesianLinearRegressor(np.zeros(D), ref.Diagonal(np.ones(D)))

        def run():
            fx = f(ref.ColVecs(X), σ2)
            return ref.posterior(fx, y), ref.logpdf(fx, y)

        return run, n, f"literal reference op sequence (posterior + logpdf as two calls), N={n} of the D={D} workload per step, scipy/OpenBLAS fp64"
    if c["kind"] == "rff":
        n = args.cpu_sample or (1 << 13)
        rng = np.random.default_rng(0)
        W, b = rng.standard_normal((D, c["din"])), rng.uniform(0, 2 * np.pi, D)
        x = rng.standard_normal((c["din"], n))
        σ2 = np.exp(rng.standard_normal(n))
        y = rng.standard_normal(n)
        bfr = ref.BasisFunctionRegressor(ref.BayesianLinearRegressor(np.zeros(D), ref.Diagonal(np.ones(D))),
                                         lambda z: ref.ColVecs(math.sqrt(2.0 / D) * np.cos(W @ z.X + b[:, None])))

        def run():
            fx = bfr(ref.ColVecs(x), σ2)
            return ref.posterior(fx, y), ref.logpdf(fx, y)

        return run, n, f"literal reference op sequence through BasisFunctionRegressor (ϕ evaluated twice, as the reference does), N={n} of the D={D} workload per step"
    n = args.cpu_sample or (1 << 15)
    rng = np.random.default_rng(0)
    B = rng.standard_normal((D, D)) / math.sqrt(D)
    post = ref.BayesianLinearRegressor(rng.standard_normal(D), B @ B.T + np.eye(D))
    Xt = np.asfortranarray(rng.standard_normal((D, n)))

    def run():
        return ref.mean_and_var(post(ref.ColVecs(Xt), 0.1))

    return run, n, f"reference mean_and_var (dpotrf + dtrsm + column norms) on N*={n} test points of the D={D} workload per step"


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (its literal op sequence on scipy/OpenBLAS --
    Julia itself is not installable here) with all host threads, on a bounded sample of the SAME config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    c = resolve(args, max(world, args.gpus))
    cores = use_all_host_threads()
    run, n, sample = cpu_pass_factory(args, c)
    for _ in range(args.warmup):
        run()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run()
    dt = (time.perf_counter() - t0) / args.steps
    value = n / dt
    print(json.dumps({
        "impl": "reference", "metric": c["metric"], "value": value, "unit": c["unit"], "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config_dict(args, c, max(world, args.gpus)),
        "cpu_baseline": {"value": value, "unit": c["unit"], "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": c["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------ our arm
class Env:
    pass


def setup(args):
    import torch

    import blr_b200 as blr

    E = Env()
    E.torch, E.blr = torch, blr
    E.rank = int(os.environ.get("RANK", "0"))
    E.world = int(os.environ.get("WORLD_SIZE", "1"))
    E.local = int(os.environ.get("LOCAL_RANK", "0"))
    if E.world != args.gpus and E.world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={E.world}")
    E.numa = {"bound": False, "why": "--no-numa-bind"} if args.no_numa_bind else bind_to_gpu_numa(E.local)
    torch.cuda.set_device(E.local)
    E.ctx = blr.Context(E.local)
    blr.set_default_context(E.ctx)
    if E.world > 1:
        import torch.distributed as dist

        # NCCL prints its version banner on stdout at communicator creation: keep stdout to the ONE JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", E.local))
            E.ctx.init_comm_from_torch()
            dist.barrier()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    E.stream = torch.cuda.ExternalStream(E.ctx.stream(), device=torch.device("cuda", E.local))
    return E


def barrier(E):
    if E.world > 1:
        E.torch.distributed.barrier()
    E.torch.cuda.synchronize()
    E.ctx.sync()


def max_over_ranks(E, v):
    if E.world == 1:
        return v
    t = E.torch.tensor([v], dtype=E.torch.float64, device="cuda")
    E.torch.distributed.all_reduce(t, op=E.torch.distributed.ReduceOp.MAX)
    return float(t.item())


def min_over_ranks(E, v):
    return -max_over_ranks(E, -v)


def timed_steps(E, args, step):
    """W warm-up steps, then exactly K steps between barrier + synchronize, CUDA events on the library's stream, max over ranks."""
    for _ in range(args.warmup):
        out = step()
    sampler = ClockSampler(E.local) if E.rank == 0 else None
    barrier(E)
    launches0 = E.ctx.launch_count()
    ev0, ev1 = E.torch.cuda.Event(enable_timing=True), E.torch.cuda.Event(enable_timing=True)
    ev0.record(E.stream)
    for _ in range(args.steps):
        out = step()
    ev1.record(E.stream)
    barrier(E)
    ms = max_over_ranks(E, ev0.elapsed_time(ev1)) / args.steps
    return ms, E.ctx.launch_count() - launches0, (sampler.stop() if sampler else None), out


def expected_key(args, c):
    k = f"{args.config}_seed{args.seed}_N{c['n']}_D{c['dim']}"
    if c["kind"] == "infer":
        k += ("_scalar" if args.scalar_noise else "") + ("_pm" if args.prior_mean != "zero" else "")
    return k


def logpdf_parity(args, c, lp):
    exp = {}
    if os.path.exists(EXPECTED_PATH):
        try:
            exp = json.load(open(EXPECTED_PATH))
        except Exception:
            exp = {}
    key = expected_key(args, c)
    if key not in exp:
        return {"checked": False, "ok": True, "key": key, "note": "no committed value for this data set; logpdf printed for pinning"}
    rel = abs(lp - exp[key]) / abs(exp[key])
    return {"checked": True, "ok": bool(rel <= 1e-11), "key": key, "rel_err": rel, "expected_logpdf": exp[key],
            "what": "log marginal likelihood vs the committed value of the same synthetic data set (independent of the number of GPUs); "
                    "the statistics behind it are Freivalds-checked at this size in tests/test_gpu_fullsize.py"}


def cublas_dgemm_tflops(torch, n=8192, reps=5):
    """Independent fp64 yardstick (SURVEY.md 8d): cuBLAS Dgemm n^3 through torch, CUDA events.  Reported next to the library's
    own DMMA issue-loop calibration; never on the product path."""
    try:
        a = torch.randn((n, n), dtype=torch.float64, device="cuda")
        b = torch.randn((n, n), dtype=torch.float64, device="cuda")
        c = torch.empty((n, n), dtype=torch.float64, device="cuda")
        torch.mm(a, b, out=c)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            torch.mm(a, b, out=c)
        e1.record()
        torch.cuda.synchronize()
        tf = 2.0 * n ** 3 * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12
        del a, b, c
        torch.cuda.empty_cache()
        return tf
    except Exception:  # e.g. out of memory next to a device-filling workload: the yardstick is optional
        return None


def roofline_block(E, args, n_loc, D, g_ms, solve_ms, ms_per_step):
    achieved = gram_flops(n_loc, D) / (g_ms * 1e-3) / 1e12
    cal = E.ctx.calibrate() if not args.no_calibrate else {}
    if cal:
        cal["cublas_dgemm_8192_tflops"] = cublas_dgemm_tflops(E.torch)
    peak = cal.get("dmma_tflops") or NOMINAL_FP64_TFLOPS
    traffic, tsrc = None, None
    if os.path.exists(TRAFFIC_PATH):
        try:
            tj = json.load(open(TRAFFIC_PATH))
            traffic, tsrc = tj.get(f"D{D}_N{n_loc}"), tj.get("_source")
        except Exception:
            traffic = None
    return {"bound": "tensor", "kernel": "gram_tma_kernel (fp64 DMMA.8x8x4 + TMA bulk copies)", "achieved": achieved, "peak": peak,
            "unit": "TFLOP/s", "frac": achieved / peak,
            "peak_source": "on-box pure-DMMA issue loop (blr_calibrate_dmma); MEASURED_PEAKS.json has no fp64 entry" if cal
            else "nominal 148 SM x 64 DFMA/clk x 1.965 GHz",
            "peak_nominal": NOMINAL_FP64_TFLOPS, "frac_of_nominal": achieved / NOMINAL_FP64_TFLOPS, "calibration": cal,
            "kernel_ms": g_ms, "solve_ms": solve_ms, "kernel_share_of_step": g_ms / ms_per_step,
            "algorithmic_flops_per_launch": gram_flops(n_loc, D), "algorithmic_bytes_per_launch": 8.0 * n_loc * (D + 2),
            "traffic": traffic, "traffic_source": tsrc if traffic is not None else "no ncu capture committed for this shape"}


def pinned_h2d_roofline(E, nbytes=1 << 30, reps=4):
    """Rank-concurrent page-locked H2D copy rate: the roofline of the e2e leg (every rank copies at the same time)."""
    torch = E.torch
    src = torch.empty(nbytes // 8, dtype=torch.float64, pin_memory=True)
    src.zero_()
    dst = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    dst.copy_(src, non_blocking=True)
    barrier(E)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(src, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    gbs = reps * nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9
    return {"per_rank_gbs_min": min_over_ranks(E, gbs), "per_rank_gbs_max": max_over_ranks(E, gbs),
            "how": f"{reps} x {nbytes >> 20} MiB cudaMemcpyAsync from page-locked memory on every rank at once, CUDA events"}


def host_budget_obs(E, bytes_per_obs, want):
    """Largest power of two <= want whose page-locked buffers (all ranks of the box) stay within ~40 % of the free host RAM."""
    try:
        import psutil

        avail = psutil.virtual_memory().available
    except Exception:  # pragma: no cover
        avail = 64 << 30
    n = want
    while n > (1 << 16) and n * bytes_per_obs * E.world > 0.4 * avail:
        n >>= 1
    return n


def fill_tiled(torch, dst, gen, block_rows=1 << 16):
    """Fill a big page-locked (rows, D) tensor with N(0,1) by tiling one random block (memcpy speed instead of RNG speed)."""
    rows = dst.shape[0]
    blk = torch.empty((min(block_rows, rows),) + tuple(dst.shape[1:]), dtype=dst.dtype)
    blk.normal_(generator=gen)
    for a in range(0, rows, blk.shape[0]):
        b = min(rows, a + blk.shape[0])
        dst[a:b].copy_(blk[: b - a])


def dump_sample(x):
    """A result array (numpy, or a torch tensor on any device) as float64 numpy for --dump-outputs: whole up to
    DUMP_MAX_ELEMS elements, else its values at fixed seeded flat positions (a function of the element count only)."""
    n = int(np.prod(x.shape))
    idx = None if n <= DUMP_MAX_ELEMS else np.unique(np.random.default_rng(0).integers(0, n, DUMP_MAX_ELEMS))
    if isinstance(x, np.ndarray):
        return np.array(x if idx is None else x.ravel()[idx], dtype=np.float64)
    import torch

    flat = x.reshape(-1)
    if idx is not None:
        flat = flat[torch.from_numpy(idx).to(x.device)]
    return flat.to(torch.float64).cpu().numpy().reshape(x.shape if idx is None else -1)


def write_dump(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ posterior + logpdf configs
def run_infer(args, E, c):
    torch, blr, ctx = E.torch, E.blr, E.ctx
    N, D = c["n"], c["dim"]
    lo, hi = blr.ShardPlan(N, E.world).bounds(E.rank)
    n_loc = hi - lo
    rff = None
    if c["kind"] == "rff":
        din = c["din"]
        rng = np.random.default_rng(0)  # the same feature map on every rank
        rff = blr.RandomFourierFeatures(rng.standard_normal((D, din)), rng.uniform(0, 2 * np.pi, D), ctx)
        X = blr.DeviceMatrix.alloc(ctx, din, n_loc).synth_(args.seed + 3, lo)
    else:
        X = blr.DeviceMatrix.alloc(ctx, D, n_loc).synth_(args.seed, lo)
    σ2 = blr.DeviceVector.alloc(ctx, n_loc)
    y = blr.DeviceVector.alloc(ctx, n_loc)
    ctx.check(ctx.lib.blr_vec_synth_noise(ctx.handle, σ2.handle, args.seed, lo))
    if c["kind"] == "rff":
        ctx.check(ctx.lib.blr_vec_synth_noise(ctx.handle, y.handle, args.seed + 6, lo))  # targets: any fixed data
    else:
        ctx.check(ctx.lib.blr_vec_synth_targets(ctx.handle, X.handle, σ2.handle, args.seed, lo, y.handle))
    ctx.sync()
    mw = np.zeros(D) if args.prior_mean == "zero" else 0.1 * np.random.default_rng(args.seed + 17).standard_normal(D)
    f = blr.BayesianLinearRegressor(mw, blr.Diagonal(np.ones(D)))
    model = blr.BasisFunctionRegressor(f, rff) if rff is not None else f
    fx = model(blr.ColVecs(X), 0.37 if args.scalar_noise else σ2)
    fx.ctx = ctx
    gram_ms, solve_ms, prep_ms = [], [], []

    def step():
        post, lp = blr.posterior_and_logpdf(fx, y)  # public API; returns m', Λ' (host) and logpdf
        t = ctx.last_timings()
        gram_ms.append(t["gram_ms"]); solve_ms.append(t["solve_ms"]); prep_ms.append(t["prep_ms"])
        return post, lp

    ms_per_step, launches, clocks, (post, lp) = timed_steps(E, args, step)
    if args.dump_outputs and E.rank == 0:
        res = post.blr if rff is not None else post
        write_dump(args.dump_outputs, {"posterior_mean": dump_sample(res.mw), "posterior_precision": dump_sample(res.Λw.dense()),
                                       "logpdf": np.float64(lp)})
    gram_ms, solve_ms, prep_ms = gram_ms[-args.steps:], solve_ms[-args.steps:], prep_ms[-args.steps:]
    out = None
    if E.rank == 0:
        g_ms = statistics.mean(gram_ms)
        extra_fl = 2.0 * N * D * c["din"] if rff is not None else 0.0
        out = {
            "metric": c["metric"], "value": N / (ms_per_step * 1e-3), "unit": c["unit"], "n_gpus": E.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config_dict(args, c, E.world), "gpu_launches": launches, "clocks": clocks,
            "roofline": roofline_block(E, args, n_loc, D, g_ms, statistics.mean(solve_ms), ms_per_step),
            "phase_ms": {"prep": statistics.mean(prep_ms), "gram": g_ms, "dxd": statistics.mean(solve_ms)},
            "path_tflops": (path_flops(N, D) + extra_fl) / (ms_per_step * 1e-3) / 1e12 / E.world,
            "logpdf": lp, "parity": logpdf_parity(args, c, lp),
        }
    del X, σ2, y, fx, post
    return out


def e2e_infer(args, E, c):
    """posterior+logpdf through the public API from page-locked HOST memory: every step uploads its observations chunk by
    chunk (H2D inside the timed region, overlapped with the Gram kernel), accumulates, all-reduces, solves, and reads back the
    posterior mean / precision / logpdf (D2H).  Each rank streams its own buffer (every GPU has its own PCIe link)."""
    torch, blr, ctx = E.torch, E.blr, E.ctx
    D = c["dim"]
    if c["kind"] == "rff":
        din = c["din"]
        n_host = host_budget_obs(E, 8 * (din + 2), min(args.e2e_obs or (1 << 22), c["n"] // E.world))
        xh = torch.empty((n_host, din), dtype=torch.float64, pin_memory=True)
        yh = torch.empty(n_host, dtype=torch.float64, pin_memory=True)
        sh = torch.empty(n_host, dtype=torch.float64, pin_memory=True)
        g = torch.Generator().manual_seed(1234 + E.rank)
        fill_tiled(torch, xh, g)
        sh.normal_(generator=g).exp_()
        yh.normal_(generator=g)
        rng = np.random.default_rng(0)
        rff = blr.RandomFourierFeatures(rng.standard_normal((D, din)), rng.uniform(0, 2 * np.pi, D), ctx)
        bfr = blr.BasisFunctionRegressor(blr.BayesianLinearRegressor(np.zeros(D), blr.Diagonal(np.ones(D))), rff)
        xn, yn, sn = xh.numpy().T, yh.numpy(), sh.numpy()

        def step():
            fx = bfr(blr.ColVecs(xn), sn)
            fx.ctx = ctx
            return blr.posterior_and_logpdf(fx, yn)

        h2d = n_host * (din + 2) * 8
    else:
        n_host = host_budget_obs(E, 8 * (D + 2), min(args.e2e_obs or (1 << 22), c["n"]))
        chunk = min(args.e2e_chunk, n_host)
        Xh = torch.empty((n_host, D), dtype=torch.float64, pin_memory=True)  # = column-major D x n_host
        yh = torch.empty(n_host, dtype=torch.float64, pin_memory=True)
        sh = torch.empty(n_host, dtype=torch.float64, pin_memory=True)
        g = torch.Generator().manual_seed(1234 + E.rank)
        fill_tiled(torch, Xh, g)
        sh.normal_(generator=g).exp_()
        yh.normal_(generator=g)
        Xn, yn, sn = Xh.numpy(), yh.numpy(), sh.numpy()
        f = blr.BayesianLinearRegressor(np.zeros(D), blr.Diagonal(np.ones(D)))

        def step():
            return blr.posterior_and_logpdf_streamed(f, Xn.T, yn, sn, chunk=chunk, ctx=ctx)

        h2d = n_host * (D + 2) * 8
    roof = pinned_h2d_roofline(E)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    barrier(E)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        post, lp = step()
    ctx.sync()
    dt = max_over_ranks(E, (time.perf_counter() - t0) / args.steps)
    gbs = h2d / dt / 1e9
    return {"value": n_host * E.world / dt, "unit": c["unit"], "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int((D * D + D + 1) * 8),
            "obs_per_step": n_host * E.world, "obs_per_rank": n_host, "steps": args.steps, "ms_per_step": dt * 1e3,
            "h2d_gbs_per_rank": gbs, "h2d_roofline": roof, "frac_of_h2d_roofline": gbs / roof["per_rank_gbs_min"], "numa": {k: v for k, v in E.numa.items() if k != "restore"},
            "note": f"each rank streams {n_host} host-resident observations of the workload per step from page-locked memory "
                    "(cost is linear in N; the leg is bound by the host->device link, whose rank-concurrent copy rate is h2d_roofline); "
                    "wall clock around the public API call, max over ranks"}


# ------------------------------------------------------------------------------------------------ cfg4: marginals + rand
def run_predict(args, E, c):
    import scipy.linalg as sl

    from blr_b200.runtime import make_noise

    torch, blr, ctx = E.torch, E.blr, E.ctx
    Nt, D, S = c["n"], c["dim"], c["samples"]
    lo, hi = blr.ShardPlan(Nt, E.world).bounds(E.rank)
    n = hi - lo
    # fit: observations sharded, one allreduce, posterior replicated on every rank
    n_fit = 1 << 20
    flo, fhi = blr.ShardPlan(n_fit, E.world).bounds(E.rank)
    Xf = blr.DeviceMatrix.alloc(ctx, D, fhi - flo).synth_(args.seed, flo)
    s2f, yf = blr.DeviceVector.alloc(ctx, fhi - flo), blr.DeviceVector.alloc(ctx, fhi - flo)
    ctx.check(ctx.lib.blr_vec_synth_noise(ctx.handle, s2f.handle, args.seed, flo))
    ctx.check(ctx.lib.blr_vec_synth_targets(ctx.handle, Xf.handle, s2f.handle, args.seed, flo, yf.handle))
    f = blr.BayesianLinearRegressor(np.zeros(D), blr.Diagonal(np.ones(D)))
    fx = f(blr.ColVecs(Xf), s2f)
    fx.ctx = ctx
    post, lp_fit = blr.posterior_and_logpdf(fx, yf)
    del Xf, s2f, yf, fx
    dpost = post._device(ctx)
    # this rank's test points (torch-owned so that the checker can read the same bytes)
    Xt = torch.empty((n, D), dtype=torch.float64, device="cuda")
    mv = torch.empty((2, n), dtype=torch.float64, device="cuda")
    Y = torch.empty((S, n), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    Xd = blr.DeviceMatrix.wrap_torch(ctx, Xt, 0).synth_(args.seed + 1, lo)
    noise, keep = make_noise(ctx, 0.1, n)

    def mean_var():
        ctx.check(ctx.lib.blr_mean_var_dev(ctx.handle, dpost.handle, Xd.handle, C.byref(noise), C.c_void_p(mv[0].data_ptr()),
                                           C.c_void_p(mv[1].data_ptr())))

    def rand():
        ctx.check(ctx.lib.blr_rand_finite_dev(ctx.handle, dpost.handle, Xd.handle, C.byref(noise), S, None, None, 7 + E.rank,
                                              C.c_void_p(Y.data_ptr())))

    dump = args.dump_outputs and E.rank == 0
    ms_mv, launches, clocks, _ = timed_steps(E, args, mean_var)
    ms_r, _, clocks_r, _ = timed_steps(E, args, rand)
    if dump:  # Y is overwritten by rand_supplied below
        outputs = {"mean": dump_sample(mv[0]), "var": dump_sample(mv[1]), "rand": dump_sample(Y)}
    # rand with SUPPLIED draws resident on the device -- the reference-parity mode (src/bayesian_linear_regression.jl:51-52: the
    # caller's RNG stream); the draws are generated once, outside the timed region (torch's generator: any N(0,1) stream will do)
    Zs = torch.randn((S, n), dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(args.seed + 99))
    torch.cuda.synchronize()

    def rand_supplied():
        ctx.check(ctx.lib.blr_rand_finite_dev(ctx.handle, dpost.handle, Xd.handle, C.byref(noise), S, None, C.c_void_p(Zs.data_ptr()),
                                              7 + E.rank, C.c_void_p(Y.data_ptr())))

    ms_rs, _, clocks_rs, _ = timed_steps(E, args, rand_supplied)
    if dump:
        outputs["rand_supplied_draws"] = dump_sample(Y)
        write_dump(args.dump_outputs, outputs)
    del Zs
    # parity on sampled blocks: x'm', |L^-1 x|² + σ² from the host posterior by torch (checker), rand with supplied draws
    Lp = np.linalg.cholesky(post.Λw.dense())
    cft, mt = torch.from_numpy(Lp).cuda(), torch.from_numpy(post.mw).cuda()
    rng = np.random.default_rng(2)
    blk = min(8192, n)
    worst = 0.0
    for a in [0, n - blk] + [int(v) for v in rng.integers(0, max(n - blk, 1), 6)]:
        Xc = Xt[a:a + blk]
        al = torch.linalg.solve_triangular(cft, Xc.T, upper=False)
        v_o, m_o = (al * al).sum(0) + 0.1, Xc @ mt
        worst = max(worst, float((mv[1, a:a + blk] - v_o).norm() / v_o.norm()), float((mv[0, a:a + blk] - m_o).norm() / m_o.norm()))
    Zw = np.asfortranarray(rng.standard_normal((D, S)))
    Zy = torch.randn((S, blk), dtype=torch.float64, device="cuda")
    Yc = torch.empty((S, blk), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    Xb = blr.DeviceMatrix.wrap_torch(ctx, Xt[:blk], 0)
    nz, kz = make_noise(ctx, 0.1, blk)
    ctx.check(ctx.lib.blr_rand_finite_dev(ctx.handle, dpost.handle, Xb.handle, C.byref(nz), S, Zw.ctypes.data_as(C.c_void_p),
                                          C.c_void_p(Zy.data_ptr()), 0, C.c_void_p(Yc.data_ptr())))
    ctx.sync()
    Wt = torch.from_numpy(post.mw[:, None] + sl.solve_triangular(Lp.T, Zw, lower=False)).cuda()
    Yo = (Xt[:blk] @ Wt).T + math.sqrt(0.1) * Zy
    worst_r = float((Yc - Yo).norm() / Yo.norm())
    finite = bool(torch.isfinite(mv).all()) and bool(torch.isfinite(Y).all())
    worst, worst_r = max_over_ranks(E, worst), max_over_ranks(E, worst_r)
    out = None
    if E.rank == 0:
        fl_mv = float(n) * D * (D + 1) + 2.0 * n * D
        fl_r = 2.0 * n * D * S + float(D) * D * S
        cal = ctx.calibrate() if not args.no_calibrate else {}
        peak = cal.get("dmma_tflops") or NOMINAL_FP64_TFLOPS
        out = {
            "metric": c["metric"], "value": Nt / (ms_mv * 1e-3), "unit": c["unit"], "n_gpus": E.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_mv, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config_dict(args, c, E.world), "gpu_launches": launches, "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "var_tma_kernel (triangular GEMM W x on DMMA.8x8x4, register column norms)",
                         "achieved": fl_mv / (ms_mv * 1e-3) / 1e12, "peak": peak, "unit": "TFLOP/s", "frac": fl_mv / (ms_mv * 1e-3) / 1e12 / peak,
                         "peak_source": "on-box pure-DMMA issue loop" if cal else "nominal", "peak_nominal": NOMINAL_FP64_TFLOPS,
                         "kernel_ms": ms_mv, "algorithmic_flops_per_launch": fl_mv, "algorithmic_bytes_per_launch": 8.0 * n * (D + 3),
                         "traffic": None},
            "rand": {"value": Nt / (ms_r * 1e-3), "unit": "points/s", "samples": S, "ms_per_step": ms_r, "clocks": clocks_r,
                     "tflops_per_gpu": fl_r / (ms_r * 1e-3) / 1e12, "frac_of_dmma_peak": fl_r / (ms_r * 1e-3) / 1e12 / peak,
                     "hbm_gbs_algorithmic_per_gpu": 8.0 * n * (D + S) / (ms_r * 1e-3) / 1e9, "draws": "device Philox4x32-10, Box-Muller"},
            "rand_supplied_draws": {"value": Nt / (ms_rs * 1e-3), "unit": "points/s", "samples": S, "ms_per_step": ms_rs, "clocks": clocks_rs,
                                    "tflops_per_gpu": fl_r / (ms_rs * 1e-3) / 1e12, "frac_of_dmma_peak": fl_r / (ms_rs * 1e-3) / 1e12 / peak,
                                    "hbm_gbs_algorithmic_per_gpu": 8.0 * n * (D + 2 * S) / (ms_rs * 1e-3) / 1e9,
                                    "draws": "N x S standard normals resident on the device (the reference's mode: the caller's RNG stream, "
                                             ":51-52); two-group kernel"},
            "fit_logpdf": lp_fit,
            "parity": {"checked": True, "ok": bool(worst < 1e-9 and worst_r < 1e-9 and finite), "marginals_max_rel_err": worst,
                       "rand_rel_err": worst_r, "finite": finite,
                       "what": "8 sampled blocks of 8192 test points per rank against torch (x'm', |L^-1 x|^2 + σ²); rand with supplied draws on one block"},
        }
    return out, post


def e2e_predict(args, E, c, post):
    torch, blr, ctx = E.torch, E.blr, E.ctx
    D = c["dim"]
    n_host = host_budget_obs(E, 8 * (D + 2), args.e2e_obs or (1 << 21))
    Xh = torch.empty((n_host, D), dtype=torch.float64, pin_memory=True)
    fill_tiled(torch, Xh, torch.Generator().manual_seed(99 + E.rank))
    Xn = Xh.numpy().T
    roof = pinned_h2d_roofline(E)

    def step():
        fx = post(blr.ColVecs(Xn), 0.1)
        fx.ctx = ctx
        return blr.mean_and_var(fx)

    for _ in range(2):
        step()
    barrier(E)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        m, v = step()
    ctx.sync()
    dt = max_over_ranks(E, (time.perf_counter() - t0) / args.steps)
    h2d = n_host * D * 8
    return {"value": n_host * E.world / dt, "unit": c["unit"], "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(2 * n_host * 8),
            "points_per_step": n_host * E.world, "steps": args.steps, "ms_per_step": dt * 1e3, "h2d_gbs_per_rank": h2d / dt / 1e9,
            "h2d_roofline": roof, "numa": {k: v for k, v in E.numa.items() if k != "restore"},
            "note": "mean_and_var(post(ColVecs(host matrix), 0.1)) through the public API: upload of the test points, kernel, download of mean and var"}


# ------------------------------------------------------------------------------------------------ driver
def run_ours(args):
    E = setup(args)
    c = resolve(args, E.world)
    post = None
    if c["kind"] == "predict":
        out, post = run_predict(args, E, c)
    else:
        out = run_infer(args, E, c)
    if not args.no_e2e:
        e2e = e2e_predict(args, E, c, post) if c["kind"] == "predict" else e2e_infer(args, E, c)
        if out is not None:
            out["e2e"] = e2e
    # CPU baseline (rank 0, N = 1 only): the reference's literal op sequence on this box's host cores, bounded sample
    if E.rank == 0 and E.world == 1 and not args.no_cpu:
        cores = use_all_host_threads(E.numa.get("restore"))
        run, n, sample = cpu_pass_factory(args, c)
        t0 = time.perf_counter()
        run()
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": n / dt, "unit": c["unit"], "cores": cores, "kind": "port", "sample": sample + ", one pass"}
    rc = 0
    if E.rank == 0:
        print(json.dumps(out))
        if not out.get("parity", {}).get("ok", True):
            sys.stderr.write(f"PARITY FAILURE: {out['parity']}\n")
            rc = 3
    if E.world > 1:
        E.torch.distributed.barrier()
        E.torch.distributed.destroy_process_group()
    sys.exit(rc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg3", choices=sorted(CONFIGS))
    ap.add_argument("--n-obs", type=int, default=0, help="override the config's N (sweeps / tools)")
    ap.add_argument("--dim", type=int, default=0, help="override the config's D (sweeps / tools)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--prior-mean", default="zero", choices=["zero", "random"],
                    help="random: non-zero prior mean, i.e. δ = y - X'mw needs a pass over X (every step of sequential conditioning)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="units in the CPU-baseline sample (default: per config)")
    ap.add_argument("--e2e-obs", type=int, default=0, help="host-resident units per rank for the e2e leg (default 2^22, bounded by host RAM)")
    ap.add_argument("--e2e-chunk", type=int, default=1 << 16)
    ap.add_argument("--max-log2-per-gpu", type=int, default=24, help="cfg4: test points per GPU are capped at 2^this")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-calibrate", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--scalar-noise", action="store_true", help="secondary measurement: Σy = σ² I instead of the headline's heteroscedastic noise")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (float64; see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
