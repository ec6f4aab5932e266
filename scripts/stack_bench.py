"""TransformStack against M separate member calls, on one GPU, timed with CUDA events.

    python scripts/stack_bench.py --out-dir DIR [--reps 5]

Config 1 (1024^2 frames, 128 px patches) and config 2 (2048^2, 256 px), float32 and float64, B in {1, 8} frames,
M in {1, 4, 16} kernels of the alpha / epsilon grid: stack.apply(x) through k2_stack and through the per-kernel
column pass (rpsf_plan_set_stack_mode) against stack[m].apply(x) for every m (each member warmed up, with its own
plans), with the bytes each path needs by a model computed from the plan's shapes and their fraction of the device
copy rate measured in the same run, a saturated sweep (a threshold that about 0.1 % of the pixels exceed) and a
masked sweep (0.01 % of the pixels masked at random), and TransformStack.construct against M x construct.  Every
timed input is a device tensor; each number is the median of --reps timed calls after two warm-up calls.  Writes
DIR/r08_stack_bench.json with the GPU's name, power limit and clocks.
"""
import argparse
import ctypes
import itertools
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import regularizepsf_b200 as rp  # noqa: E402
from oracle import cpu_oracle as oracle  # noqa: E402

CONFIGS = {"config1": ((1024, 1024), 128), "config2": ((2048, 2048), 256)}
PAIRS = list(itertools.product((0.5, 1.0, 2.0, 3.0), (0.3, 0.1, 0.05, 0.01)))


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [v.strip() for v in line.split(",")]))
    except Exception as exc:  # the measurement still stands; say why the context is missing
        return {"error": str(exc)}


def timed(torch, fn, reps):
    for _ in range(2):
        fn()
    times = []
    for _ in range(reps):
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        fn()
        end.record()
        end.synchronize()
        times.append(start.elapsed_time(end))
    return float(np.median(times))


def copy_rate(torch):
    """Device-to-device copy rate of a 2 GiB buffer, GB/s (bytes read + written over time)."""
    a = torch.empty(1 << 31, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    ms = timed(torch, lambda: b.copy_(a), 5)
    return 2 * a.numel() / (ms * 1e-3) / 1e9


def byte_model(lib, stack, dtype, h, w, b):
    """Bytes one stack.apply of b frames moves (fused, per-kernel), from the plan's shapes: K1 reads the frames and
    writes the row bands; the column pass reads the bands (once, or once per kernel), each kernel's tile per frame and
    writes the spectra; the overlap-add reads every spectrum and writes every output frame."""
    import torch
    ns = stack._native[(dtype, torch.cuda.current_device())]
    plan = next(reversed(ns._plans.values()))
    info = (ctypes.c_int64 * 9)()
    lib.rpsf_plan_info(plan, info)
    m, p = len(stack), stack.psf_shape[0]
    rs = 4 if dtype == "float32" else 8
    spec = info[0] * p * (p // 2) * 2 * rs                 # one frame's spectra for one kernel
    bands = (info[2] - m * ns._plans_batch[plan] * spec) // ns._plans_batch[plan]
    kern = len(stack.coordinates) * (p * (p // 2) + p) * 2 * rs
    frame = h * w * rs
    k1, k3 = b * (frame + bands), m * b * (spec + frame)
    fused = k1 + b * (bands + m * (spec + kern)) + k3
    per_kernel = k1 + m * b * (bands + spec + kern) + k3
    return fused, per_kernel


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    os.makedirs(args.out_dir, exist_ok=True)
    result = {"gpu": gpu_info(), "reps": args.reps, "unit": "ms per call (median of CUDA-event timings)", "apply": [],
              "saturated": [], "masked": [], "construct": []}
    rng = np.random.default_rng(0)
    lib = rp._native.load()
    rate = copy_rate(torch)
    result["copy_rate_GBps"] = rate
    print("copy rate", rate, "GB/s", flush=True)
    for name, (shape, size) in CONFIGS.items():
        coords = rp.calculate_covering(shape, size)
        src = oracle.coma_psf_cube(coords, size, shape)
        tgt = oracle.gaussian_psf_cube(len(coords), size, 3.0)
        source, target = rp.ArrayPSF(rp.IndexedCube(coords, src)), rp.ArrayPSF(rp.IndexedCube(coords, tgt))
        full = rp.TransformStack.construct(source, target, [a for a, _ in PAIRS], [e for _, e in PAIRS])
        frames = torch.from_numpy(rng.normal(100.0, 20.0, (8,) + shape)).cuda()
        for m in (1, 4, 16):
            alphas, epsilons = [a for a, _ in PAIRS[:m]], [e for _, e in PAIRS[:m]]
            t_stack = timed(torch, lambda: rp.TransformStack.construct(source, target, alphas, epsilons), args.reps)
            t_loop = timed(torch, lambda: [rp.ArrayPSFTransform.construct(source, target, a, e)
                                           for a, e in zip(alphas, epsilons)], args.reps)
            cube = len(coords) * size * size * 16              # complex128: the PSF cubes are float64
            result["construct"].append({"config": name, "M": m, "stack_ms": t_stack, "loop_ms": t_loop,
                                        "model_bytes_stack": (2 + m) * cube, "model_bytes_loop": 3 * m * cube,
                                        "copy_fraction_stack": (2 + m) * cube / (t_stack * 1e-3) / 1e9 / rate})
            print(json.dumps(result["construct"][-1]), flush=True)
        for dtype in ("float32", "float64"):
            want = torch.float32 if dtype == "float32" else torch.float64
            for b in (1, 8):
                x = frames[:b].to(want).contiguous()
                for m in (1, 4, 16):
                    stack = rp.TransformStack(coords, full.kernels[:m])
                    members = [stack[k] for k in range(m)]
                    t_stack = timed(torch, lambda: stack.apply(x, dtype=dtype), args.reps)
                    stack._stack_mode = 1
                    t_per = timed(torch, lambda: stack.apply(x, dtype=dtype), args.reps)
                    stack._stack_mode = 0
                    t_loop = timed(torch, lambda: [tr.apply(x, dtype=dtype) for tr in members], args.reps)
                    fused_b, per_b = byte_model(lib, stack, dtype, shape[0], shape[1], b)
                    row = {"config": name, "dtype": dtype, "B": b, "M": m, "stack_ms": t_stack,
                           "per_kernel_ms": t_per, "loop_ms": t_loop, "speedup": t_loop / t_stack,
                           "k2_stack_vs_per_kernel": t_per / t_stack, "model_bytes_fused": fused_b,
                           "model_bytes_per_kernel": per_b,
                           "copy_fraction_fused": fused_b / (t_stack * 1e-3) / 1e9 / rate,
                           "copy_fraction_per_kernel": per_b / (t_per * 1e-3) / 1e9 / rate}
                    result["apply"].append(row)
                    print(json.dumps(row), flush=True)
                    del stack, members
                    torch.cuda.empty_cache()
        # saturated and masked sweeps: float32, one frame, 16 kernels
        x = frames[:1].float().contiguous()
        threshold = float(torch.quantile(x[0].flatten()[:1 << 24].double(), 0.999))
        mask = torch.from_numpy(rng.random(shape) < 1e-4).cuda()
        stack = rp.TransformStack(coords, full.kernels)
        members = [stack[k] for k in range(len(stack))]
        for key, kw in (("saturated", {"saturation_threshold": threshold}), ("masked", {"mask": mask})):
            t_stack = timed(torch, lambda: stack.apply(x, **kw), args.reps)
            t_loop = timed(torch, lambda: [tr.apply(x, **kw) for tr in members], args.reps)
            row = {"config": name, "dtype": "float32", "B": 1, "M": len(stack), "stack_ms": t_stack, "loop_ms": t_loop,
                   "speedup": t_loop / t_stack}
            if key == "saturated":
                row["threshold"] = threshold
            result[key].append(row)
            print(key, json.dumps(row), flush=True)
        del stack, members, full
        torch.cuda.empty_cache()
    path = os.path.join(args.out_dir, "r08_stack_bench.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
