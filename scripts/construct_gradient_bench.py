#!/usr/bin/env python
"""The gradient of construct (the transfer kernel of two PSFs) and of the PSF FFT cube, and a fitting step through them.

    python scripts/construct_gradient_bench.py --out-dir DIR [--iters N] [--rounds R]

Writes DIR/construct_gradient_bench.json (one JSON line) and prints it.  Configurations: config 2 (2048^2, 256-px patches,
289 patches) and config 1 (1024^2, 128-px patches) in float32 (complex64 cubes), config 2 in float64; coma source ->
Gaussian target PSF, random incoming gradients.  Reported in us per call, CUDA events over N calls after a warm-up,
median of R rounds:
- construct forward (rpsf_construct_kernel), the construct VJP (rpsf_construct_kernel_backward with both cube outputs and
  grad_alpha / grad_eps) and the FFT VJP (rpsf_psf_fft2_adjoint of the source cube);
- each as a fraction of the HBM copy rate measured in the same run (a 4 GiB device-to-device copy), from the bytes the
  algorithm must move, counted from the shapes: the forward reads S and T and writes K (3 cubes); the VJP reads G, S and
  T and writes grad_S and grad_T (5 cubes); the FFT VJP reads G and writes the real values (1.5 cubes; its complex
  scratch cube, written by the row pass and read by the column pass, is not counted);
- one fitting step on 8 frames: `reconstruct -> apply -> MSE -> backward`, with the source values, alpha and epsilon
  requiring grad, and the same step with a fresh `construct` per step (new native transform and plans every step).
A config-2 complex64 cube is 151.5 MB, beyond the 126 MB L2; a config-1 cube (38 MB) is not.  The device name and power
limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import regularizepsf_b200 as rp  # noqa: E402
from oracle import cpu_oracle as oracle  # noqa: E402
from regularizepsf_b200 import _native  # noqa: E402
from scripts.kernel_gradient_bench import copy_peak_bytes_per_s, device_info, time_calls  # noqa: E402


def make_psfs(shape, patch, real):
    coords = [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, patch)]
    source = torch.from_numpy(oracle.coma_psf_cube(coords, patch, shape)).cuda().to(real)
    target = torch.from_numpy(oracle.gaussian_psf_cube(len(coords), patch, 3.0)).cuda().to(real)
    return coords, source, target


def rounds_of(fn, iters, rounds, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    return [time_calls(fn, iters) for _ in range(rounds)]


def run_kernels(name, shape, patch, dtype, iters, rounds, warmup, peak):
    real = torch.float32 if dtype == "float32" else torch.float64
    cplx = torch.complex64 if dtype == "float32" else torch.complex128
    code = _native.F32 if dtype == "float32" else _native.F64
    lib = _native.load()
    coords, sv, tv = make_psfs(shape, patch, real)
    n = len(coords)
    s = rp.ArrayPSF(rp.DeviceCube(coords, sv)).fft_cube.tensor
    t = rp.ArrayPSF(rp.DeviceCube(coords, tv)).fft_cube.tensor
    g = torch.randn(s.shape, dtype=cplx, device=s.device)
    k, gs, gt = torch.empty_like(s), torch.empty_like(s), torch.empty_like(s)
    ae = torch.empty(2, dtype=torch.float64, device=s.device)
    xv = torch.empty_like(sv)
    stream = _native.current_stream_ptr(torch)

    def forward():
        _native.check(lib.rpsf_construct_kernel(s.data_ptr(), t.data_ptr(), k.data_ptr(), s.numel(), code, 1.0, 0.1, 0,
                                                stream))

    def vjp():
        _native.check(lib.rpsf_construct_kernel_backward(s.data_ptr(), t.data_ptr(), g.data_ptr(), s.numel(), code, 1.0,
                                                         0.1, gs.data_ptr(), gt.data_ptr(), ae.data_ptr(), 0, stream))

    def fft_vjp():
        _native.check(lib.rpsf_psf_fft2_adjoint(g.data_ptr(), xv.data_ptr(), n, patch, code, 0, stream))

    cube = s.numel() * s.element_size()
    out = {"config": name, "shape": list(shape), "patch": patch, "dtype": dtype, "patches": n, "cube_bytes": cube}
    for label, fn, nbytes in (("construct_forward", forward, 3 * cube), ("construct_vjp", vjp, 5 * cube),
                              ("fft_vjp", fft_vjp, 3 * cube // 2)):
        us = rounds_of(fn, iters, rounds, warmup)
        med = statistics.median(us)
        out[label] = {"us": round(med, 2), "rounds": [round(v, 2) for v in us], "bytes": nbytes,
                      "fraction_of_copy_peak": round(nbytes / (med * 1e-6) / peak, 3)}
    return out


def run_fit_step(name, shape, patch, dtype, frames, iters, rounds, warmup):
    real = torch.float32 if dtype == "float32" else torch.float64
    coords, sv, tv = make_psfs(shape, patch, real)
    sv.requires_grad_()
    alpha = torch.tensor(1.0, dtype=torch.float64, device="cuda", requires_grad=True)
    epsilon = torch.tensor(0.1, dtype=torch.float64, device="cuda", requires_grad=True)
    source, target = rp.ArrayPSF(rp.DeviceCube(coords, sv)), rp.ArrayPSF(rp.DeviceCube(coords, tv))
    x = torch.from_numpy(np.stack([oracle.starfield(shape, seed=s) for s in range(frames)])).cuda().to(real)
    with torch.no_grad():
        y = rp.ArrayPSFTransform.construct(source, target, 1.2, 0.15).apply(x, dtype=dtype)
    transform = rp.ArrayPSFTransform.construct(source, target, alpha, epsilon)

    def clear():
        sv.grad = alpha.grad = epsilon.grad = None

    def reconstruct_step():
        clear()
        transform.reconstruct(source, target, alpha, epsilon)
        torch.nn.functional.mse_loss(transform.apply(x, dtype=dtype), y).backward()

    def fresh_step():
        clear()
        fresh = rp.ArrayPSFTransform.construct(source, target, alpha, epsilon)
        torch.nn.functional.mse_loss(fresh.apply(x, dtype=dtype), y).backward()

    r_us, f_us = [], []
    for _ in range(warmup):
        reconstruct_step(); fresh_step()
    torch.cuda.synchronize()
    for _ in range(rounds):
        r_us.append(time_calls(reconstruct_step, iters))
        f_us.append(time_calls(fresh_step, iters))
    r, f = statistics.median(r_us), statistics.median(f_us)
    return {"config": name, "shape": list(shape), "patch": patch, "dtype": dtype, "frames": frames,
            "requires_grad": ["source values", "alpha", "epsilon"],
            "reconstruct_step_us": round(r, 1), "fresh_construct_step_us": round(f, 1),
            "reconstruct_rounds": [round(v, 1) for v in r_us], "fresh_construct_rounds": [round(v, 1) for v in f_us]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("construct_gradient_bench needs a CUDA device")
    torch.cuda.set_device(0)
    peak = copy_peak_bytes_per_s()
    result = {"device": device_info(), "copy_peak_GB_per_s": round(peak / 1e9, 1), "iters": args.iters,
              "rounds": args.rounds, "kernels": [], "fit_step": []}
    cfgs = [("config2", (2048, 2048), 256, "float32"), ("config1", (1024, 1024), 128, "float32"),
            ("config2", (2048, 2048), 256, "float64")]
    for name, shape, patch, dtype in cfgs:
        result["kernels"].append(run_kernels(name, shape, patch, dtype, args.iters, args.rounds, args.warmup, peak))
    for name, shape, patch, dtype in cfgs:
        iters = args.iters if dtype == "float32" else max(args.iters // 4, 2)
        result["fit_step"].append(run_fit_step(name, shape, patch, dtype, 8, iters, args.rounds, args.warmup))
    result["device"]["after"] = device_info()["power_limit_and_max_sm_clock"]
    line = json.dumps(result)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "construct_gradient_bench.json"), "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
