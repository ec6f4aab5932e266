#!/usr/bin/env python
"""Eager calls against CUDA graph replays of the same calls: device-resident apply and a whole fitting step.

    python scripts/graph_bench.py [--out profiles/r05_graph_bench.json] [--iters N] [--rounds R]

Rows (float32, random transfer kernels for apply; coma source -> Gaussian target PSFs for the fitting step):
- apply of one 512^2 frame at 32 px, one 1024^2 frame at 128 px, and config 2 (2048^2, 256 px) with 1 and 8 frames;
- the fitting step `reconstruct -> apply -> MSE -> backward -> Adam(capturable=True).step()` with the source values,
  alpha and epsilon requiring grad, at config 1 (1024^2, 128 px, 8 frames) and config 2 (2048^2, 256 px, 8 frames);
- the kernel layout (rpsf_transform_set_kernel) alone at config 1 and 2: what a captured call of a transform with a
  trainable kernel adds to each replay, since it lays the kernel out in the graph.
"eager_never_captured" times the eager apply before its transform was captured, "eager" after (every call waits for
the transform's event then).  Each row is timed over warm shapes, N calls per round, median of R rounds, three ways: CUDA events around the N calls
(device_us), a host clock around the N calls and a final synchronise (wall_us), and the host clock until the last call
returns, before the synchronise (host_us: what the caller's thread spends issuing).  The inputs are the same tensors at
every call, so a working set below the 126 MB L2 (the 512^2 and 1024^2 rows) is read from L2.  The device name and
power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

import regularizepsf_b200 as rp  # noqa: E402
from oracle import cpu_oracle as oracle  # noqa: E402
from regularizepsf_b200 import _native  # noqa: E402
from scripts.kernel_gradient_bench import device_info  # noqa: E402


def timed(fn, iters, rounds):
    """(device_us, wall_us, host_us) per call, medians over rounds."""
    dev, wall, host = [], [], []
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        start.record()
        for _ in range(iters):
            fn()
        stop.record()
        t1 = time.perf_counter()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        dev.append(start.elapsed_time(stop) * 1e3 / iters)
        wall.append((t2 - t0) * 1e6 / iters)
        host.append((t1 - t0) * 1e6 / iters)
    return {"device_us": round(statistics.median(dev), 2), "wall_us": round(statistics.median(wall), 2),
            "host_us": round(statistics.median(host), 2)}


def capture(fn, warmup=3):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warmup):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        fn()
    torch.cuda.synchronize()
    return graph


def apply_row(name, hw, patch, frames, iters, rounds):
    coords = [tuple(int(v) for v in c) for c in rp.calculate_covering((hw, hw), patch)]
    g = torch.Generator(device="cuda").manual_seed(1)
    kernel = torch.randn((len(coords), patch, patch), dtype=torch.complex64, device="cuda", generator=g)
    t = rp.ArrayPSFTransform(rp.DeviceCube(coords, kernel))
    x = torch.rand((frames, hw, hw) if frames > 1 else (hw, hw), device="cuda", generator=g)
    eager = lambda: t.apply(x)                                         # noqa: E731
    for _ in range(3):
        eager()
    never_captured = timed(eager, iters, rounds)
    graph = capture(eager)
    for _ in range(3):
        eager()
        graph.replay()
    return {"row": name, "frames": frames, "eager_never_captured": never_captured, "eager": timed(eager, iters, rounds),
            "replay": timed(graph.replay, iters, rounds)}


class Fit:
    def __init__(self, hw, patch, frames):
        coords = [tuple(int(v) for v in c) for c in rp.calculate_covering((hw, hw), patch)]
        src = torch.from_numpy(oracle.coma_psf_cube(coords, patch, (hw, hw))).cuda().float()
        tgt = torch.from_numpy(oracle.gaussian_psf_cube(len(coords), patch, 3.0)).cuda().float()
        self.values = src.clone().requires_grad_()
        self.alpha = torch.tensor(1.2, dtype=torch.float64, device="cuda", requires_grad=True)
        self.epsilon = torch.tensor(0.15, dtype=torch.float64, device="cuda", requires_grad=True)
        self.source = rp.ArrayPSF(rp.DeviceCube(coords, self.values))
        self.target = rp.ArrayPSF(rp.DeviceCube(coords, tgt))
        self.target.fft_cube
        g = torch.Generator(device="cuda").manual_seed(3)
        self.x = torch.rand((frames, hw, hw), device="cuda", generator=g)
        ref = rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.DeviceCube(coords, src)), self.target, 1.0, 0.1)
        self.y = ref.apply(self.x).detach()
        self.transform = rp.ArrayPSFTransform.construct(self.source, self.target, 1.2, 0.15)
        self.opt = torch.optim.Adam([self.values, self.alpha, self.epsilon], lr=1e-4, capturable=True)

    def step(self):
        self.transform.reconstruct(self.source, self.target, self.alpha, self.epsilon)
        loss = ((self.transform.apply(self.x) - self.y) ** 2).mean()
        loss.backward()
        self.opt.step()

    def eager_step(self):
        self.opt.zero_grad(set_to_none=True)
        self.step()


def fit_row(name, hw, patch, frames, iters, rounds):
    eager = Fit(hw, patch, frames)
    for _ in range(3):
        eager.eager_step()
    eager_t = timed(eager.eager_step, iters, rounds)
    del eager
    fit = Fit(hw, patch, frames)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fit.eager_step()
    torch.cuda.current_stream().wait_stream(side)
    fit.opt.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        fit.step()
    torch.cuda.synchronize()
    for _ in range(3):
        graph.replay()
    # the kernel layout a captured call of a trainable kernel adds to each replay
    nt = next(iter(fit.transform._native.values()))
    kt = fit.transform._kernel_on(torch, 0)
    stream = _native.current_stream_ptr(torch)
    layout = timed(lambda: nt.set_kernel(kt, stream), iters, rounds)
    return {"row": name, "frames": frames, "eager": eager_t, "replay": timed(graph.replay, iters, rounds),
            "kernel_layout": layout}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_graph_bench.json"))
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("graph_bench needs a CUDA device")
    torch.cuda.set_device(0)
    rows = [apply_row("apply 512^2 / 32 px", 512, 32, 1, args.iters, args.rounds),
            apply_row("apply 1024^2 / 128 px", 1024, 128, 1, args.iters, args.rounds),
            apply_row("apply config 2 (2048^2 / 256 px)", 2048, 256, 1, args.iters, args.rounds),
            apply_row("apply config 2 (2048^2 / 256 px)", 2048, 256, 8, args.iters, args.rounds),
            fit_row("fitting step config 1 (1024^2 / 128 px)", 1024, 128, 8, max(args.iters // 5, 5), args.rounds),
            fit_row("fitting step config 2 (2048^2 / 256 px)", 2048, 256, 8, max(args.iters // 5, 5), args.rounds)]
    result = {"device": device_info(), "iters": args.iters, "rounds": args.rounds, "rows": rows}
    line = json.dumps(result)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
