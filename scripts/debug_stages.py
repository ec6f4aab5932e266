"""GPU debugging aid: check K1, K1+K2 and the full apply stage by stage against numpy/scipy.

K1 leaves the row bands (each frame row transformed once per corner column, without the row window); what a patch
reads of them is checked through K1+K2, whose output is the per-patch spectrum at the start of the workspace."""
import ctypes
import sys
import os

import numpy as np
import scipy.fft

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from oracle import cpu_oracle as oracle
import regularizepsf_b200 as rp
from regularizepsf_b200 import _native


def run(shape, P, dtype_name="float32", pad_mode="symmetric"):
    coords = [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, P)]
    src = oracle.coma_psf_cube(coords, P, shape)
    tgt = oracle.gaussian_psf_cube(len(coords), P, 3.0)
    image = oracle.starfield(shape, seed=5).astype(np.float64)
    K = oracle.transfer_kernel(oracle.psf_fft(src), oracle.psf_fft(tgt), 1.0, 0.1)
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, K))
    nt = t._native_transform(dtype_name)
    H, W = shape
    plan = nt.plan(H, W, _native.PAD_MODES[pad_mode], 0, H, 1)
    info = nt.plan_info(plan)
    lib = nt.lib
    tdt = torch.float32 if dtype_name == "float32" else torch.float64
    npdt = np.float32 if dtype_name == "float32" else np.float64
    cdt = np.complex64 if dtype_name == "float32" else np.complex128
    img_d = torch.from_numpy(image.astype(npdt)).cuda()
    out_d = torch.zeros((H, W), dtype=tdt, device="cuda")
    n = info["active_patches"]
    assert n == len(coords), (n, len(coords))

    def stage(k):
        """The workspace after the first k kernels: (patch spectra (n, P, P/2), row bands (rows, P/2))."""
        _native.check(lib.rpsf_apply_stages(plan, img_d.data_ptr(), W, H * W, 0, H, out_d.data_ptr(), W, H * W, 0, 1,
                                            k, 0))
        ptr, nbytes = ctypes.c_void_p(), ctypes.c_int64()
        _native.check(lib.rpsf_plan_workspace(plan, ctypes.byref(ptr), ctypes.byref(nbytes)))
        host = np.empty(nbytes.value // np.dtype(cdt).itemsize, dtype=cdt)
        _native.check(lib.rpsf_copy_to_host(host.ctypes.data, ptr, nbytes.value, 0))
        return host[:n * P * (P // 2)].reshape(n, P, P // 2), host[n * P * (P // 2):].reshape(-1, P // 2)

    # reference intermediates in float64
    padded = np.pad(image, ((2 * P, 2 * P), (2 * P, 2 * P)), mode=pad_mode)
    win = oracle.apodization((P, P))
    patches = np.stack([padded[r + 2 * P:r + 3 * P, c + 2 * P:c + 3 * P] for r, c in coords]) * win
    scale = np.abs(image).max()

    # K1: every band row is the unwindowed row spectrum times 2 of some frame row; each such spectrum is a row of
    # some patch before the row window, so the set of band rows must be found among them
    w1 = np.sin((np.arange(P) + 0.5) * np.pi / P)
    X1 = 2 * scipy.fft.rfft(patches / w1[None, :, None], axis=-1)          # row spectra, no row window, times 2
    ref = np.concatenate([X1[..., :1].real + 1j * X1[..., P // 2:P // 2 + 1].real, X1[..., 1:P // 2]], axis=-1)
    ref = ref.reshape(-1, P // 2)
    _, bands = stage(1)
    live = bands[np.abs(bands).max(axis=1) > 0]
    nearest = np.array([np.abs(ref - row).max(axis=1).min() for row in live[:: max(1, len(live) // 256)]])
    print(f"[P={P} {dtype_name}] K1 band rows: {len(live)} non-zero, err {nearest.max()/scale:.2e} (rel to max)")

    X2 = scipy.fft.fft2(patches)
    Y = X2 * K
    y_full = scipy.fft.ifft2(Y)                       # complex, (n,P,P)
    Uc = scipy.fft.fft(np.real(y_full), axis=-1) / P  # row spectra of the real output (K2 leaves the row 1/P to the folded 1/P^2)
    got2, _ = stage(2)
    e_main = np.abs(got2[:, :, 1:] - Uc[:, :, 1:P // 2]).max()
    e_dc = np.abs(got2[:, :, 0].real - Uc[:, :, 0].real).max()
    e_ny = np.abs(got2[:, :, 0].imag - Uc[:, :, P // 2].real).max()
    print(f"[P={P} {dtype_name}] K2 err main {e_main/scale:.2e} dc {e_dc/scale:.2e} nyq {e_ny/scale:.2e}")

    stage(3)
    torch.cuda.synchronize()
    want = oracle.apply_transform(image, coords, K, pad_mode=pad_mode)
    got = out_d.cpu().numpy()
    print(f"[P={P} {dtype_name}] apply err {np.abs(got - want).max()/scale:.2e}  info={info}")


if __name__ == "__main__":
    run((96, 80), 32)
    run((96, 80), 32, "float64")
    run((48, 40), 16)
    run((192, 160), 64)
    run((300, 260), 128)
    run((520, 600), 256)
    run((520, 600), 256, "float64")
    run((1100, 1030), 512)
    run((1100, 1030), 512, "float64")
