#!/usr/bin/env python
"""logpdf against logpdf_and_grad (blr_logpdf_grad) on the device, with every gradient and without dX, timed with CUDA events on
the library's stream; the grad_x kernel time from a separate torch.profiler run and its achieved rate 2 N D² / kernel time
against blr_calibrate_dmma measured in the same process.  One JSON line per shape, with the card name and its power limit.

With --k 1,8,32 it measures blr_logpdf_multi_grad instead, one line per shape and k: the call with every gradient for an (N, k)
Y, the rank-k grad_x kernel from torch.profiler and its rate 2 N D (D + k) / kernel time against blr_calibrate_dmma, and, for
comparison, blr_logpdf_grad called once per column (timed once).

    python tools/bench_grad.py [--reps 5] [--k 1,8,32] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import blr_b200 as blr  # noqa: E402

SHAPES = [(1 << 20, 256), (1 << 22, 1024)]  # cfg2 and the large-D shape
NO_DX = ("y", "σ²", "mw", "Λw")


def power_limit():
    r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "unknown"


def timed(ctx, st, fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(reps):
        out = fn()
    e1.record(st)
    ctx.sync()
    torch.cuda.synchronize()
    del out
    return e0.elapsed_time(e1) / reps


def bench_multi(ctx, st, fx, y, N, D, k, reps, dmma):
    from torch.profiler import ProfilerActivity, profile

    y0 = torch.as_tensor(y.download(), device="cuda")
    Y = torch.stack([y0 * (1.0 + 0.01 * j) for j in range(k)], dim=1)  # (N, k)
    multi = lambda: blr.logpdf_and_grad(fx, Y)  # noqa: E731
    multi()
    ctx.sync()
    ms = timed(ctx, st, multi, reps)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            out = multi()
        ctx.sync()
        torch.cuda.synchronize()
    del out
    kms = float("nan")
    for ev in prof.key_averages():
        if "grad_x_tma_kernel<true>" in ev.key:
            tot = getattr(ev, "self_device_time_total", None) or getattr(ev, "self_cuda_time_total", 0.0)
            kms = tot / ev.count / 1e3  # us -> ms per launch
    tf = 2.0 * N * D * (D + k) / (kms * 1e-3) / 1e12
    cols = [blr.DeviceVector.wrap_torch(ctx, Y[:, j].contiguous()) for j in range(k)]

    def single():
        for c in cols:  # each result dropped before the next call: dX alone is N D doubles
            blr.logpdf_and_grad(fx, c)

    single_ms = timed(ctx, st, single, 1)
    return {"tool": "bench_grad", "N": N, "D": D, "k": k, "multi_grad_ms": ms, "grad_x_multi_kernel_ms": kms,
            "grad_x_multi_tflops": tf, "dmma_tflops": dmma, "grad_x_multi_share_of_dmma": tf / dmma,
            "single_grad_k_calls_ms": single_ms, "reps": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--k", default=None, help="comma-separated column counts: measure blr_logpdf_multi_grad")
    args = ap.parse_args()
    ctx = blr.Context(0)
    blr.set_default_context(ctx)
    dmma = ctx.calibrate()["dmma_tflops"]
    card, plim = torch.cuda.get_device_name(0), power_limit()
    st = torch.cuda.ExternalStream(ctx.stream())
    lines = []
    for N, D in SHAPES:
        X = blr.DeviceMatrix.alloc(ctx, D, N).synth_(0)
        s2, y = blr.DeviceVector.alloc(ctx, N), blr.DeviceVector.alloc(ctx, N)
        ctx.check(ctx.lib.blr_vec_synth_noise(ctx.handle, s2.handle, 0, 0))
        ctx.check(ctx.lib.blr_vec_synth_targets(ctx.handle, X.handle, s2.handle, 0, 0, y.handle))
        rng = np.random.default_rng(1)
        f = blr.BayesianLinearRegressor(0.1 * rng.standard_normal(D), blr.Diagonal(np.exp(rng.standard_normal(D))))
        Xt = X.as_torch()  # (N, D): gradients come back as device tensors
        fx = f(blr.ColVecs(Xt), s2)
        if args.k:
            for k in (int(v) for v in args.k.split(",")):
                line = bench_multi(ctx, st, fx, y, N, D, k, args.reps, dmma)
                line.update({"device": card, "power_limit": plim})
                print(json.dumps(line), flush=True)
                lines.append(line)
            del X, Xt, fx, s2, y
            torch.cuda.empty_cache()
            continue
        runs = {"logpdf": lambda: blr.logpdf(fx, y), "grad_all": lambda: blr.logpdf_and_grad(fx, y),
                "grad_no_dX": lambda: blr.logpdf_and_grad(fx, y, wrt=NO_DX)}
        ms = {}
        for name, fn in runs.items():
            fn()
            ctx.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(args.reps):
                out = fn()
            e1.record(st)
            ctx.sync()
            torch.cuda.synchronize()
            ms[name] = e0.elapsed_time(e1) / args.reps
            del out
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                out = blr.logpdf_and_grad(fx, y)
            ctx.sync()
            torch.cuda.synchronize()
        del out
        kms = float("nan")
        for k in prof.key_averages():
            if "grad_x_tma_kernel" in k.key:
                tot = getattr(k, "self_device_time_total", None) or getattr(k, "self_cuda_time_total", 0.0)
                kms = tot / k.count / 1e3  # us -> ms per launch
        tf = 2.0 * N * D * D / (kms * 1e-3) / 1e12
        line = {"tool": "bench_grad", "N": N, "D": D, "logpdf_ms": ms["logpdf"], "grad_all_ms": ms["grad_all"],
                "grad_no_dX_ms": ms["grad_no_dX"], "grad_x_kernel_ms": kms, "grad_x_tflops": tf, "dmma_tflops": dmma,
                "grad_x_share_of_dmma": tf / dmma, "device": card, "power_limit": plim, "reps": args.reps}
        print(json.dumps(line), flush=True)
        lines.append(line)
        del X, Xt, fx, s2, y
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
