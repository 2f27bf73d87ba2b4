#!/usr/bin/env python
"""Throughput of noise-vector refinement (ganrev_refine_l2: Adam on ||G(z) - x||^2 through G's tensor-core backward pass).

Workloads: 65,536 32x32 faces x 100 iterations and 8192 3x64x64 faces x 50 iterations (nd = 100, apply_r.lua's noiseDim), with
x = G(z*) and z0 = z* + 0.5 N(0,1) -- the refinement of a rough guess.  Prints one JSON line: image-iterations/s, the time of one
iteration over the time of one forward pass of G on the same faces, per-kernel CUDA-event time and executed TFLOP/s of a separate
profiled run (5 iterations), a PyTorch-CPU autograd + Adam stand-in on a small sample (thread count stated), and the GPU's name,
power limit and SM clocks read in the same call.  Needs a B200; there is no CPU path for the measured numbers.

--masked: each workload also runs as face completion (ganrev_refine_masked_l2) with a centred H/2 x W/2 hole in every face, timed
alternately with the unmasked call in the same process (three pairs, the best of each reported), plus its own profiled run.
Without the flag the output is unchanged.
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
from __graft_entry__ import load_package  # noqa: E402

WORKLOADS = [(1, 32, 32, 100, 65536, 100), (3, 64, 64, 100, 8192, 50)]   # C, H, W, nd, faces, iterations


def gpu_info(gpu):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", str(gpu), f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [s.strip() for s in out.strip().split(",")]))


def timed(ctx, fn):
    ctx.sync()
    t0 = time.perf_counter()
    fn()
    ctx.sync()
    return time.perf_counter() - t0


def cpu_standin(pkg, C, H, W, nd, n, iters):
    import torch
    from oracle import torch_grad
    p = pkg.weights.unpack(pkg.weights.init_G(C, H, W, nd, seed=1), pkg.weights.g_layout(C, H, W, nd))
    rng = np.random.default_rng(5)
    z = torch.from_numpy(rng.normal(size=(n, nd)).astype(np.float32)).requires_grad_(True)
    x = torch.from_numpy(rng.random(size=(n, C, H, W)).astype(np.float32))
    opt = torch.optim.Adam([z], lr=0.01)
    t0 = time.perf_counter()
    for _ in range(iters):
        opt.zero_grad()
        torch_grad.objective(p, C, H, W, nd, z, x, 0.0).sum().backward()
        opt.step()
    dt = time.perf_counter() - t0
    return {"what": "PyTorch-CPU fp32 autograd through G + torch.optim.Adam (a stand-in, not the library)", "threads": torch.get_num_threads(),
            "geometry": [C, H, W, nd], "faces": n, "iterations": iters, "image_iterations_per_sec": n * iters / dt}


def profiled(ctx, run, iters):
    ctx.profile_reset(); ctx.profile_enable(True)
    run()
    ctx.profile_enable(False)
    return {k: {"launches": v["launches"], "ms_per_iteration": v["ms"] / iters,
                "tflops_executed": v["flops"] / max(v["ms"], 1e-9) / 1e9, "gbs": v["bytes"] / max(v["ms"], 1e-9) / 1e6}
            for k, v in ctx.profile().items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpu", type=int, default=0)
    ap.add_argument("--scale", type=float, default=1.0, help="multiply the face counts (quick runs)")
    ap.add_argument("--cpu-faces", type=int, default=8)
    ap.add_argument("--cpu-iters", type=int, default=2)
    ap.add_argument("--masked", action="store_true", help="also time the masked refinement (centre hole), alternated with the unmasked")
    a = ap.parse_args()
    pkg = load_package()
    ctx = pkg.Context(a.gpu)
    res = {"metric": "refine_image_iterations_per_sec", "unit": "image-iterations/s", "gpu": gpu_info(a.gpu), "workloads": []}
    for C, H, W, nd, N, iters in WORKLOADS:
        N = max(1, int(N * a.scale))
        ctx.load_G(C, H, W, nd, pkg.weights.init_G(C, H, W, nd, seed=1))
        rng = np.random.default_rng(3)
        zs = rng.normal(size=(N, nd)).astype(np.float32)
        z0 = (zs + 0.5 * rng.normal(size=zs.shape)).astype(np.float32)
        x = ctx.forward_G(zs)
        ctx.refine_l2(1, x[:min(N, 4096)], z0[:min(N, 4096)], iters=2, want_attrs=False, want_fixed=False)   # builds the backward layers, warms every shape
        ctx.buffer_put(pkg._lib.BUF_NOISE, z0)
        t_fwd = min(timed(ctx, lambda: ctx.forward_G(None, N=N, want_images=False)) for _ in range(3))
        ctx.buffer_put(pkg._lib.BUF_IMAGES, x)
        _, _, l2_0 = ctx.refine_l2(1, None, z0, iters=0, N=N, want_attrs=False, want_fixed=False)
        t_ref = timed(ctx, lambda: ctx.refine_l2(1, None, z0, iters=iters, N=N, want_attrs=False, want_fixed=False))
        _, _, l2_1 = ctx.refine_l2(1, None, z0, iters=iters, N=N, want_attrs=False, want_fixed=False)
        t_iter = (t_ref - t_fwd) / iters            # the call ends with one forward pass + L2 of z_final
        prof_iters = min(iters, 5)
        kernels = profiled(ctx, lambda: ctx.refine_l2(1, None, z0, iters=prof_iters, N=N, want_attrs=False, want_fixed=False), prof_iters)
        res["workloads"].append({
            "geometry": [C, H, W, nd], "faces": N, "iterations": iters,
            "image_iterations_per_sec": N * iters / (t_ref - t_fwd), "call_s": t_ref, "forward_s": t_fwd,
            "iteration_over_forward": t_iter / t_fwd, "median_l2_before": float(np.median(l2_0)), "median_l2_after": float(np.median(l2_1)),
            "profiled_iterations": prof_iters, "kernels": kernels})
        if a.masked:
            mask = np.ones((N, C, H, W), np.uint8)
            mask[:, :, H // 4:H // 4 + H // 2, W // 4:W // 4 + W // 2] = 0
            ctx.buffer_put(pkg._lib.BUF_MASK, mask)
            unmasked = lambda: ctx.refine_l2(1, None, z0, iters=iters, N=N, want_attrs=False, want_fixed=False)
            masked = lambda: ctx.refine_masked_l2(1, None, None, z0, iters=iters, N=N, want_attrs=False, want_fixed=False)
            ctx.refine_masked_l2(1, None, None, z0[:min(N, 4096)], iters=2, N=min(N, 4096), want_attrs=False, want_fixed=False)
            t_u, t_m = [], []
            for _ in range(3):
                t_u.append(timed(ctx, unmasked))
                t_m.append(timed(ctx, masked))
            _, _, l2_m = ctx.refine_masked_l2(1, None, None, z0, iters=iters, N=N, want_attrs=False, want_fixed=False)
            res["workloads"][-1]["masked"] = {
                "mask": "centred H/2 x W/2 hole", "call_s_unmasked": t_u, "call_s_masked": t_m,
                "image_iterations_per_sec_unmasked": N * iters / (min(t_u) - t_fwd),
                "image_iterations_per_sec_masked": N * iters / (min(t_m) - t_fwd),
                "masked_over_unmasked_time": (min(t_m) - t_fwd) / (min(t_u) - t_fwd),
                "median_masked_l2_after": float(np.median(l2_m)),
                "kernels": profiled(ctx, lambda: ctx.refine_masked_l2(1, None, None, z0, iters=prof_iters, N=N, want_attrs=False,
                                                                      want_fixed=False), prof_iters)}
    res["value"] = res["workloads"][0]["image_iterations_per_sec"]
    res["cpu_standin"] = cpu_standin(pkg, 1, 32, 32, 100, a.cpu_faces, a.cpu_iters)
    res["gpu_after"] = gpu_info(a.gpu)
    ctx.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
