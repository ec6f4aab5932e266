#!/usr/bin/env python
"""Forward (apply) against transpose (apply_adjoint) on device-resident frames, and loss.backward() end to end.

    python scripts/adjoint_bench.py --out-dir DIR [--iters N] [--rounds R]

Writes DIR/adjoint_bench.json (one JSON line) and prints it.  Configurations: config 2 (2048^2, 256-px patches) and
config 1 (1024^2, 128-px patches), coma source -> Gaussian target PSF, 8 and 1 frames per call, float32; config 2 in
float64; then `loss = (apply(x) * w).sum(); loss.backward()` at config 2.  Times are CUDA events over N calls after a
warm-up, forward and adjoint alternated R times (the median round is reported), in us per frame.  At 8 frames per call
the working set (frames, 606 MB of spectra) is far beyond the 126 MB L2.  A separate pass with the plans' per-stage
events splits each call into K1 / K2 / K3 and the rest (for the adjoint: the copy into the box and the fold).
`bytes` are what each stage must move at least, from the shapes.  The device name and power limit are read in the
same run.
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


def make_transform(shape, patch):
    coords = [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, patch)]
    source = rp.ArrayPSF(rp.IndexedCube(coords, oracle.coma_psf_cube(coords, patch, shape)))
    target = rp.ArrayPSF(rp.IndexedCube(coords, oracle.gaussian_psf_cube(len(coords), patch, 3.0)))
    return rp.ArrayPSFTransform.construct(source, target, 1.0, 0.1), coords


def time_calls(fn, iters):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) * 1e3 / iters          # us per call


def stage_split(nt, plan, fn, iters):
    """K1 / K2 / K3 us per call from the plan's events, and the whole call, in one run with the events on."""
    lib = nt.lib
    lib.rpsf_plan_enable_timing(plan, 1)
    ms, calls = (ctypes.c_double * 3)(), ctypes.c_int()
    lib.rpsf_plan_read_timing(plan, ms, ctypes.byref(calls))          # reset
    total = time_calls(fn, iters)
    lib.rpsf_plan_read_timing(plan, ms, ctypes.byref(calls))
    lib.rpsf_plan_enable_timing(plan, 0)
    k = [ms[i] * 1e3 / max(calls.value, 1) for i in range(3)]
    return {"k1": k[0], "k2": k[1], "k3": k[2], "call": total, "rest": total - sum(k)}


def traffic(shape, patch, n_patches, box, rs):
    """Least bytes per frame of each stage (read + write), from shapes."""
    h, w = shape
    spectra = n_patches * patch * (patch // 2) * 2 * rs
    kernel = n_patches * patch * (patch // 2 + 1) * 2 * rs
    fwd = {"k1": h * w * rs + spectra, "k2": 2 * spectra + kernel, "k3": spectra + h * w * rs}
    hb, wb = box
    adj = {"copy": 2 * h * w * rs, "k1": hb * wb * rs + spectra, "k2": 2 * spectra + kernel,
           "k3": spectra + hb * wb * rs, "fold": hb * wb * rs + h * w * rs}
    return {"forward": fwd, "adjoint": adj, "forward_total": sum(fwd.values()), "adjoint_total": sum(adj.values())}


def run_config(name, shape, patch, dtype, batches, iters, rounds, warmup):
    t, coords = make_transform(shape, patch)
    want = torch.float32 if dtype == "float32" else torch.float64
    rs = 4 if dtype == "float32" else 8
    frames = torch.from_numpy(np.stack([oracle.starfield(shape, seed=s) for s in range(max(batches))])).cuda().to(want)
    rows = np.array([c[0] for c in coords]); cols = np.array([c[1] for c in coords])
    box = (int(rows.max() + patch - rows.min()), int(cols.max() + patch - cols.min()))
    out = {"config": name, "shape": list(shape), "patch": patch, "dtype": dtype, "patches": len(coords),
           "box": list(box), "bytes_per_frame": traffic(shape, patch, len(coords), box, rs), "batches": {}}
    for b in batches:
        x = frames[:b].contiguous()
        fwd = lambda: t.apply(x, dtype=dtype)                         # noqa: E731
        adj = lambda: t.apply_adjoint(x, dtype=dtype)                 # noqa: E731
        for _ in range(warmup):
            fwd(); adj()
        torch.cuda.synchronize()
        f_us, a_us = [], []
        for _ in range(rounds):
            f_us.append(time_calls(fwd, iters) / b)
            a_us.append(time_calls(adj, iters) / b)
        nt = t._native_transform(dtype)
        split = {"forward": stage_split(nt, nt.plan(shape[0], shape[1], 0, 0, shape[0], b), fwd, iters),
                 "adjoint": stage_split(nt, nt.plan(shape[0], shape[1], 0, 0, shape[0], b, adjoint=True), adj, iters)}
        f, a = statistics.median(f_us), statistics.median(a_us)
        out["batches"][str(b)] = {
            "forward_us_per_frame": round(f, 2), "adjoint_us_per_frame": round(a, 2), "ratio": round(a / f, 3),
            "forward_rounds": [round(v, 2) for v in f_us], "adjoint_rounds": [round(v, 2) for v in a_us],
            "stages_us_per_call": {k: {s: round(v, 2) for s, v in d.items()} for k, d in split.items()}}
    return out


def run_backward(shape, patch, batch, iters, rounds, warmup):
    t, _ = make_transform(shape, patch)
    x = torch.from_numpy(np.stack([oracle.starfield(shape, seed=s) for s in range(batch)])).cuda().requires_grad_()
    w = torch.randn_like(x)

    def step():
        x.grad = None
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
    return {"shape": list(shape), "patch": patch, "frames": batch, "dtype": "float32",
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
        sys.exit("adjoint_bench needs a CUDA device")
    torch.cuda.set_device(0)
    result = {"device": device_info(), "iters": args.iters, "rounds": args.rounds, "configs": []}
    result["configs"].append(run_config("config2", (2048, 2048), 256, "float32", (8, 1), args.iters, args.rounds, args.warmup))
    result["configs"].append(run_config("config1", (1024, 1024), 128, "float32", (8, 1), args.iters, args.rounds, args.warmup))
    result["configs"].append(run_config("config2", (2048, 2048), 256, "float64", (8,), max(args.iters // 4, 2), args.rounds,
                                        args.warmup))
    result["backward"] = run_backward((2048, 2048), 256, 8, args.iters, args.rounds, args.warmup)
    result["device"]["after"] = device_info()["power_limit_and_max_sm_clock"]
    line = json.dumps(result)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "adjoint_bench.json"), "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
