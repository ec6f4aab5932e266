#!/usr/bin/env python
"""The gradient of apply with respect to the transfer kernel (transfer_kernel_gradient) on device-resident frames.

    python scripts/kernel_gradient_bench.py --out-dir DIR [--iters N] [--rounds R]

Writes DIR/kernel_gradient_bench.json (one JSON line) and prints it.  Configurations: config 2 (2048^2, 256-px patches)
and config 1 (1024^2, 128-px patches), coma source -> Gaussian target PSF, 8 and 1 frames per call, float32; config 2
in float64.  Reported in us per frame: the forward (apply), transfer_kernel_gradient, and `loss = (apply(x) * w).sum();
loss.backward()` with the kernel requiring grad (config 2, 8 frames, float32).  Times are CUDA events over N calls after
a warm-up, forward and gradient alternated R times (the median round is reported).  A separate pass with the forward
plan's per-stage events splits a gradient call into K1 of the image, the copy of the output gradient plus K1 of the box,
and the zeroing plus kgrad.  kgrad's algorithmic bytes come from the shapes: both spectra of every frame (2 S per
frame) and one write of the (N, P, P) complex cube per call; divided by kgrad's time they are reported as a fraction of
the HBM copy rate measured in the same run (a 4 GiB device-to-device copy).  At 8 frames per call the spectra (606 MB at
config 2) are far beyond the 126 MB L2.  The device name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import regularizepsf_b200 as rp  # noqa: E402
from oracle import cpu_oracle as oracle  # noqa: E402


def make_transform(shape, patch, trainable=False):
    coords = [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, patch)]
    source = rp.ArrayPSF(rp.IndexedCube(coords, oracle.coma_psf_cube(coords, patch, shape)))
    target = rp.ArrayPSF(rp.IndexedCube(coords, oracle.gaussian_psf_cube(len(coords), patch, 3.0)))
    t = rp.ArrayPSFTransform.construct(source, target, 1.0, 0.1)
    if trainable:
        t = rp.ArrayPSFTransform(rp.DeviceCube(coords, t._transfer_kernel.tensor.clone().requires_grad_()))
    return t, coords


def time_calls(fn, iters):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) * 1e3 / iters          # us per call


def copy_peak_bytes_per_s():
    """HBM rate of a 4 GiB device-to-device copy (read + write bytes over time), median of 5."""
    a = torch.empty(1 << 30, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    torch.cuda.synchronize()
    rates = [2 * a.numel() * 4 / (time_calls(lambda: b.copy_(a), 10) * 1e-6) for _ in range(5)]
    del a, b
    torch.cuda.empty_cache()
    return statistics.median(rates)


def stage_split(nt, plan, fn, iters):
    """us per call of the three parts of a gradient call, from the forward plan's events, and the whole call."""
    lib = nt.lib
    lib.rpsf_plan_enable_timing(plan, 1)
    ms, calls = (ctypes.c_double * 3)(), ctypes.c_int()
    lib.rpsf_plan_read_timing(plan, ms, ctypes.byref(calls))          # reset
    total = time_calls(fn, iters)
    lib.rpsf_plan_read_timing(plan, ms, ctypes.byref(calls))
    lib.rpsf_plan_enable_timing(plan, 0)
    k = [ms[i] * 1e3 / max(calls.value, 1) for i in range(3)]
    return {"k1_image": k[0], "copy_and_k1_grad": k[1], "zero_and_kgrad": k[2], "call": total, "rest": total - sum(k)}


def run_config(name, shape, patch, dtype, batches, iters, rounds, warmup, peak):
    t, coords = make_transform(shape, patch)
    want = torch.float32 if dtype == "float32" else torch.float64
    rs = 4 if dtype == "float32" else 8
    frames = torch.from_numpy(np.stack([oracle.starfield(shape, seed=s) for s in range(max(batches))])).cuda().to(want)
    grads = torch.randn_like(frames)
    out = {"config": name, "shape": list(shape), "patch": patch, "dtype": dtype, "patches": len(coords), "batches": {}}
    for b in batches:
        x, g = frames[:b].contiguous(), grads[:b].contiguous()
        fwd = lambda: t.apply(x, dtype=dtype)                                   # noqa: E731
        grad = lambda: t.transfer_kernel_gradient(x, g, dtype=dtype)            # noqa: E731
        for _ in range(warmup):
            fwd(); grad()
        torch.cuda.synchronize()
        f_us, g_us = [], []
        for _ in range(rounds):
            f_us.append(time_calls(fwd, iters) / b)
            g_us.append(time_calls(grad, iters) / b)
        nt = t._native_transform(dtype)
        plan = nt.plan(shape[0], shape[1], 0, 0, shape[0], b)
        active = nt.plan_info(plan)["active_patches"]
        split = stage_split(nt, plan, grad, iters)
        spectra = active * patch * (patch // 2) * 2 * rs
        kgrad_bytes = 2 * spectra * b + len(coords) * patch * patch * 2 * rs
        f, gr = statistics.median(f_us), statistics.median(g_us)
        out["batches"][str(b)] = {
            "forward_us_per_frame": round(f, 2), "kernel_gradient_us_per_frame": round(gr, 2), "ratio": round(gr / f, 3),
            "forward_rounds": [round(v, 2) for v in f_us], "kernel_gradient_rounds": [round(v, 2) for v in g_us],
            "stages_us_per_call": {k: round(v, 2) for k, v in split.items()},
            "kgrad_bytes_per_call": kgrad_bytes,
            "kgrad_fraction_of_copy_peak": round(kgrad_bytes / (split["zero_and_kgrad"] * 1e-6) / peak, 3)}
    return out


def run_backward(shape, patch, batch, iters, rounds, warmup):
    t, _ = make_transform(shape, patch, trainable=True)
    kernel = t._kernel_tensor
    x = torch.from_numpy(np.stack([oracle.starfield(shape, seed=s) for s in range(batch)])).cuda()
    w = torch.randn_like(x)

    def step():
        kernel.grad = None
        loss = (t.apply(x) * w).sum()
        loss.backward()

    def fwd_only():
        with torch.no_grad():
            (t.apply(x) * w).sum()

    for _ in range(warmup):
        step(); fwd_only()
    torch.cuda.synchronize()
    s_us, f_us = [], []
    for _ in range(rounds):
        s_us.append(time_calls(step, iters) / batch)
        f_us.append(time_calls(fwd_only, iters) / batch)
    s, f = statistics.median(s_us), statistics.median(f_us)
    return {"shape": list(shape), "patch": patch, "frames": batch, "dtype": "float32", "kernel_requires_grad": True,
            "forward_and_backward_us_per_frame": round(s, 2), "forward_only_us_per_frame": round(f, 2),
            "ratio": round(s / f, 3)}


def device_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as exc:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {exc}"
    return info


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("kernel_gradient_bench needs a CUDA device")
    torch.cuda.set_device(0)
    peak = copy_peak_bytes_per_s()
    result = {"device": device_info(), "copy_peak_GB_per_s": round(peak / 1e9, 1), "iters": args.iters,
              "rounds": args.rounds, "configs": []}
    result["configs"].append(run_config("config2", (2048, 2048), 256, "float32", (8, 1), args.iters, args.rounds,
                                        args.warmup, peak))
    result["configs"].append(run_config("config1", (1024, 1024), 128, "float32", (8, 1), args.iters, args.rounds,
                                        args.warmup, peak))
    result["configs"].append(run_config("config2", (2048, 2048), 256, "float64", (8,), max(args.iters // 4, 2),
                                        args.rounds, args.warmup, peak))
    result["backward"] = run_backward((2048, 2048), 256, 8, args.iters, args.rounds, args.warmup)
    result["device"]["after"] = device_info()["power_limit_and_max_sm_clock"]
    line = json.dumps(result)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "kernel_gradient_bench.json"), "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
