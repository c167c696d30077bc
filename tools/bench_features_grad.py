#!/usr/bin/env python
"""The feature-map VJP (blr_x_features_vjp) at cfg5's per-GPU share (N = 2^19 inputs, D = 4096 features) for d_in in {8, 32, 128}:
the forward blr_x_features call, the VJP for each activation (every output), torch float64 autograd forward + backward of the
same map with its peak memory, and blr_logpdf_grad with and without the VJP that follows it (d_in = 32).  Call times come from
CUDA events on the library's stream; with --profile a separate run takes kernel times from torch.profiler.  Each line carries
the card name, its power limit and blr_calibrate_dmma of the same process, the flop and byte counts from the shapes, and the
share of the bound that applies: max(6 N D d_in / DMMA rate, 8 N D / 7.7 TB/s) for the VJP (three contractions, dΦ read once
per kernel that needs it), 2 N D d_in / DMMA rate against 8 N D / 7.7 TB/s for the forward.

    python tools/bench_features_grad.py [--reps 3] [--profile] [--out FILE]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import blr_b200 as blr  # noqa: E402
from blr_b200 import _lib as L  # noqa: E402

N, D = 1 << 19, 4096
DINS = (8, 32, 128)
HBM = 7.7e12  # B/s, data sheet


def power_limit():
    r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "unknown"


def timed(ctx, st, fn, reps):
    fn()
    ctx.sync()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(reps):
        out = fn()
    e1.record(st)
    ctx.sync()
    torch.cuda.synchronize()
    del out
    return e0.elapsed_time(e1) / reps


def bound_ms(flop, nbytes, dmma_tflops):
    t_c, t_m = flop / (dmma_tflops * 1e12), nbytes / HBM
    return max(t_c, t_m) * 1e3, ("dmma" if t_c >= t_m else "hbm")


def setup(ctx, din):
    rng = np.random.default_rng(din)
    W = rng.standard_normal((D, din)) / math.sqrt(din)
    b = rng.uniform(0, 2 * math.pi, D)
    x = blr.DeviceMatrix.alloc(ctx, din, N).synth_(1)
    dphi = blr.DeviceMatrix.alloc(ctx, D, N).synth_(2)
    return W, b, x, dphi


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--profile", action="store_true", help="kernel times from torch.profiler instead of call times")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = blr.Context(0)
    blr.set_default_context(ctx)
    dmma = ctx.calibrate()["dmma_tflops"]
    card, plim = torch.cuda.get_device_name(0), power_limit()
    st = torch.cuda.ExternalStream(ctx.stream())
    lines = []

    def emit(line):
        line.update({"tool": "bench_features_grad", "device": card, "power_limit": plim, "dmma_tflops": dmma, "N": N, "D": D})
        print(json.dumps(line), flush=True)
        lines.append(line)

    for din in DINS:
        W, b, x, dphi = setup(ctx, din)
        Wf, bf = np.asfortranarray(W), np.ascontiguousarray(b)
        pW, pb = Wf.ctypes.data_as(L.c_double_p), bf.ctypes.data_as(L.c_double_p)
        dW, db = np.empty((D, din), order="F"), np.empty(D)
        dx = blr.DeviceMatrix.alloc(ctx, din, N)
        dptr, dld = dphi.device_ptr()
        xptr, xld = dx.device_ptr()

        def forward(act=0, scale=math.sqrt(2.0 / D)):
            import ctypes as C

            h = C.c_void_p()
            ctx.check(ctx.lib.blr_x_features(ctx.handle, x.handle, pW, pb, D, act, scale, C.byref(h)))
            return blr.DeviceMatrix(ctx, h, D, N, L.COLVECS)

        def vjp(act, want=("W", "b", "xin")):
            import ctypes as C

            ctx.check(ctx.lib.blr_x_features_vjp(ctx.handle, x.handle, pW, pb, D, act, 0.5, C.c_void_p(dptr), dld,
                                                 dW.ctypes.data_as(C.c_void_p) if "W" in want else None,
                                                 db.ctypes.data_as(C.c_void_p) if "b" in want else None,
                                                 C.c_void_p(xptr) if "xin" in want else None, xld))

        if args.profile:
            from torch.profiler import ProfilerActivity, profile

            forward()
            vjp(0)
            ctx.sync()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.reps):
                    out = forward()
                    del out
                    vjp(0)
                ctx.sync()
                torch.cuda.synchronize()
            k = {}
            for ev in prof.key_averages():
                for name in ("features_kernel", "features_vjp_w_kernel", "features_vjp_x_kernel", "features_vjp_reduce_kernel"):
                    if name in ev.key:
                        tot = getattr(ev, "self_device_time_total", None) or getattr(ev, "self_cuda_time_total", 0.0)
                        k[name + "_ms"] = tot / ev.count / 1e3
            emit({"d_in": din, "act": "cos", "profile": True, **k})
            del x, dphi, dx
            torch.cuda.empty_cache()
            continue

        fwd_flop, fwd_bytes = 2.0 * N * D * din, 8.0 * N * D
        ms = timed(ctx, st, forward, args.reps)
        bms, bname = bound_ms(fwd_flop, fwd_bytes, dmma)
        emit({"d_in": din, "what": "forward blr_x_features (cos)", "ms": ms, "flop": fwd_flop, "bytes": fwd_bytes, "bound": bname,
              "bound_ms": bms, "share_of_bound": bms / ms})
        fwd_ms = ms
        # dΦ is read by each of the two kernels; dW / db / dx writes are negligible
        vflop, vbytes = 6.0 * N * D * din, 2 * 8.0 * N * D
        for act, code in blr.AffineFeatures.ACTS.items():
            ms = timed(ctx, st, lambda: vjp(code), args.reps)
            bms, bname = bound_ms(vflop, vbytes, dmma)
            emit({"d_in": din, "what": f"vjp {act} (W, b, xin)", "ms": ms, "vs_forward": ms / fwd_ms, "flop": vflop, "bytes": vbytes,
                  "bound": bname, "bound_ms": bms, "share_of_bound": bms / ms})
        for want in (("W", "b"), ("xin",)):
            ms = timed(ctx, st, lambda: vjp(0, want), args.reps)
            emit({"d_in": din, "what": f"vjp cos ({', '.join(want)})", "ms": ms, "vs_forward": ms / fwd_ms})

        # torch autograd of the same map, fp64, on torch's stream
        xt = x.as_torch()  # (N, d_in)
        gt = dphi.as_torch()  # (N, D)
        Wt = torch.tensor(W, device="cuda", requires_grad=True)
        bt = torch.tensor(b, device="cuda", requires_grad=True)
        xg = xt.clone().requires_grad_(True)
        torch.cuda.synchronize()
        scale = math.sqrt(2.0 / D)

        def torch_fb():
            phi = scale * torch.cos(xg @ Wt.T + bt)
            return torch.autograd.grad(phi, (xg, Wt, bt), gt)

        torch_fb()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.reps):
            out = torch_fb()
            del out
        e1.record()
        torch.cuda.synchronize()
        peak = (torch.cuda.max_memory_allocated() - base) / 2**30
        tms = e0.elapsed_time(e1) / args.reps
        fwd_vjp = timed(ctx, st, lambda: (forward(), vjp(0)), args.reps)
        emit({"d_in": din, "what": "torch autograd forward + backward (cos, fp64)", "ms": tms, "peak_extra_GiB": peak,
              "library_forward_plus_vjp_ms": fwd_vjp, "speedup": tms / fwd_vjp})
        del xt, gt, xg, Wt, bt
        torch.cuda.empty_cache()

        if din == 32:
            phi = forward()
            rng = np.random.default_rng(3)
            s2, y = blr.DeviceVector.alloc(ctx, N), blr.DeviceVector.alloc(ctx, N)
            ctx.check(ctx.lib.blr_vec_synth_noise(ctx.handle, s2.handle, 0, 0))
            ctx.check(ctx.lib.blr_vec_synth_targets(ctx.handle, phi.handle, s2.handle, 0, 0, y.handle))
            del phi
            torch.cuda.empty_cache()
            f = blr.BayesianLinearRegressor(0.1 * rng.standard_normal(D), blr.Diagonal(np.exp(rng.standard_normal(D))))
            fx = blr.BasisFunctionRegressor(f, blr.RandomFourierFeatures(W, b))(blr.ColVecs(x), s2)
            yt = torch.as_tensor(y.download(), device="cuda")  # a CUDA y keeps ∂ℓ/∂ϕ(x) on the device in both calls
            ms_x = timed(ctx, st, lambda: blr.logpdf_and_grad(fx, yt, wrt=("X",)), 1)
            ms_w = timed(ctx, st, lambda: blr.logpdf_and_grad(fx, yt, wrt=("W", "b")), 1)
            emit({"d_in": din, "what": "logpdf_and_grad through RFF: wrt X (forward + blr_logpdf_grad) vs wrt W, b (+ VJP)",
                  "grad_dphi_ms": ms_x, "grad_W_b_ms": ms_w, "vjp_share": (ms_w - ms_x) / ms_w})
        del x, dphi, dx
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
