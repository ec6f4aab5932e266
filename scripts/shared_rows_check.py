"""Write the outputs of a fixed set of seeded calls, so that two builds can be compared bit for bit.

    python scripts/shared_rows_check.py --dump DIR

The calls cover what reads the row pass's output: 1024^2 / 128 px, 2048^2 / 256 px with 1 and 8 frames, 8192^2 /
512 px, float64, the adjoint, the kernel gradient, a saturated frame, a masked frame and an embedded 100-px patch size.
Each lands in DIR/<name>.npy; compare two directories with --compare A B (np.array_equal per file).
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _transform(torch, rp, shape, patch, seed, cdtype):
    from regularizepsf_b200.device import DeviceCube
    coords = [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, patch)]
    g = torch.Generator(device="cuda").manual_seed(seed)
    kernel = torch.randn((len(coords), patch, patch), dtype=cdtype, device="cuda", generator=g)
    return rp.ArrayPSFTransform(DeviceCube(coords, kernel))


def _frames(torch, shape, n, seed, dtype):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.rand((n,) + shape, dtype=dtype, device="cuda", generator=g) * 1000.0


def dump(out_dir: str) -> None:
    import torch
    import regularizepsf_b200 as rp
    os.makedirs(out_dir, exist_ok=True)
    f32, f64, c64, c128 = torch.float32, torch.float64, torch.complex64, torch.complex128
    results = {}
    t1 = _transform(torch, rp, (1024, 1024), 128, 1, c64)
    results["config1"] = t1.apply(_frames(torch, (1024, 1024), 8, 11, f32))
    t2 = _transform(torch, rp, (2048, 2048), 256, 2, c64)
    x2 = _frames(torch, (2048, 2048), 8, 12, f32)
    results["config2_b1"] = t2.apply(x2[:1])
    results["config2_b8"] = t2.apply(x2)
    results["config2_reflect"] = t2.apply(x2[:2], pad_mode="reflect")
    results["config2_adjoint"] = t2.apply_adjoint(x2[:2])
    results["config2_kernel_gradient"] = t2.transfer_kernel_gradient(x2[:2], x2[2:4])
    sat = x2[:1].clone()
    sat[0, 900:940, 1000:1060] = 1e5
    results["config2_saturated"] = t2.apply(sat, saturation_threshold=5e4)
    mask = torch.zeros((1, 2048, 2048), dtype=torch.bool, device="cuda")
    mask[0, 300:330, 500:520] = True
    mask[0, 1700, 17] = True
    results["config2_masked"] = t2.apply(x2[:1], mask=mask)
    t2d = _transform(torch, rp, (2048, 2048), 256, 3, c128)
    results["config2_float64"] = t2d.apply(_frames(torch, (2048, 2048), 2, 13, f64))
    t4 = _transform(torch, rp, (8192, 8192), 512, 4, c64)
    results["config4"] = t4.apply(_frames(torch, (8192, 8192), 1, 14, f32))
    te = _transform(torch, rp, (600, 520), 100, 5, c64)
    results["embedded_100"] = te.apply(_frames(torch, (600, 520), 2, 15, f32))
    torch.cuda.synchronize()
    for name, value in results.items():
        np.save(os.path.join(out_dir, name + ".npy"), value.cpu().numpy())
    print(f"wrote {len(results)} outputs to {out_dir}")


def compare(a: str, b: str) -> int:
    names = sorted(f for f in os.listdir(a) if f.endswith(".npy"))
    bad = 0
    for name in names:
        x, y = np.load(os.path.join(a, name)), np.load(os.path.join(b, name))
        same = x.shape == y.shape and np.array_equal(x, y)
        diff = "" if same or x.shape != y.shape else f" max|diff| {np.max(np.abs(x.astype(np.complex128) - y)):.3e}"
        print(f"{name:34s} {'equal' if same else 'DIFFERENT'}{diff}")
        bad += not same
    return 1 if bad or not names else 0


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--dump", metavar="DIR")
    ap.add_argument("--compare", nargs=2, metavar=("A", "B"))
    args = ap.parse_args()
    if args.dump:
        dump(args.dump)
    if args.compare:
        return compare(*args.compare)
    return 0


if __name__ == "__main__":
    sys.exit(main())
