"""Cost of apply(mask=) and of its transpose and gradients, in microseconds per frame (CUDA events).

For config 2 (2048^2 frames, 256 px patches) and config 1 (1024^2, 128 px), 8 frames and 1, float32 and float64, and
masks covering 0.01 %, 0.1 % and 1 % of the pixels plus bad columns: plain apply, masked apply, masked apply_adjoint,
the image backward and the kernel gradient of a masked apply; and, from a torch.profiler pass of its own, the ordered
fill (sat_fill) and the transposed fill (sat_fill_adjoint) alone.  Writes DIR/masked_apply_bench.json with the card's
name and power limit.

    python scripts/masked_apply_bench.py --out-dir DIR [--iters 20]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import regularizepsf_b200 as rp  # noqa: E402
from oracle import cpu_oracle as oracle  # noqa: E402

CONFIGS = {"config2": (2048, 256), "config1": (1024, 128)}
COVER = (1e-4, 1e-3, 1e-2)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as exc:  # pragma: no cover - depends on the host
        return f"unknown ({exc})"


def timed(torch, fn, iters):
    fn()
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) * 1e3 / iters


def kernel_us(torch, fn, names):
    """Device time of the kernels whose name starts with each of ``names``, for one call of ``fn`` (profiler pass)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    totals = dict.fromkeys(names, 0.0)
    for ev in prof.events():
        for name in names:
            if ev.name.split("<")[0].split("(")[0].endswith(name) and ev.device_time > 0:
                totals[name] += ev.device_time
    return totals


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    import torch
    rows = []
    for cname, (n, size) in CONFIGS.items():
        coords = [tuple(int(v) for v in c) for c in rp.calculate_covering((n, n), size)]
        kernel = oracle.gaussian_psf_cube(len(coords), size, 3.0)
        spec = np.fft.fft2(kernel)
        for batch in (8, 1):
            frames = np.stack([oracle.starfield((n, n), seed=s) for s in range(batch)])
            for dtype in ("float32", "float64"):
                real, cplx = (torch.float32, torch.complex64) if dtype == "float32" else (torch.float64, torch.complex128)
                kt = torch.from_numpy(spec).to("cuda", cplx).requires_grad_()
                t = rp.ArrayPSFTransform(rp.DeviceCube(coords, kt))
                x = torch.from_numpy(frames).to("cuda", real)
                g = torch.randn_like(x)
                with torch.no_grad():
                    plain = timed(torch, lambda: t.apply(x, dtype=dtype), args.iters) / batch
                for cover in COVER + ("columns",):
                    rng = np.random.default_rng(1)
                    if cover == "columns":
                        m = np.zeros((n, n), bool)
                        m[:, rng.choice(n, 16, replace=False)] = True
                    else:
                        m = rng.random((n, n)) < cover
                    mask = torch.from_numpy(m).cuda()
                    row = {"config": cname, "frames": batch, "dtype": dtype, "mask": cover,
                           "masked_fraction": float(m.mean()), "plain_apply_us": plain}
                    with torch.no_grad():
                        row["masked_apply_us"] = timed(torch, lambda: t.apply(x, mask=mask, dtype=dtype), args.iters) / batch
                        row["masked_adjoint_us"] = timed(
                            torch, lambda: t.apply_adjoint(g, mask=mask, dtype=dtype), args.iters) / batch
                        row["kernel_gradient_us"] = timed(
                            torch, lambda: t.transfer_kernel_gradient(x, g, mask=mask, dtype=dtype), args.iters) / batch
                    xg = x.clone().requires_grad_()
                    kt.requires_grad_(False)

                    def image_backward():
                        torch.autograd.grad(t.apply(xg, mask=mask, dtype=dtype), xg, g)
                    row["image_backward_us"] = timed(torch, image_backward, args.iters) / batch
                    kt.requires_grad_(True)
                    with torch.no_grad():
                        fwd = kernel_us(torch, lambda: t.apply(x, mask=mask, dtype=dtype), ["sat_fill"])
                        adj = kernel_us(torch, lambda: t.apply_adjoint(g, mask=mask, dtype=dtype),
                                        ["sat_fill_count", "sat_fill_adjoint", "mask_gather_adjoint"])
                    row["ordered_fill_us"] = fwd["sat_fill"] / batch
                    row["transposed_fill_us"] = adj["sat_fill_adjoint"] / batch
                    row["fill_count_us"] = adj["sat_fill_count"] / batch
                    row["gather_us"] = adj["mask_gather_adjoint"] / batch
                    rows.append(row)
                    print(json.dumps(row), flush=True)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "masked_apply_bench.json"), "w") as f:
        json.dump({"card": card(), "iters": args.iters, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
