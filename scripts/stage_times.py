"""Per-stage device times of apply() on config 2 (device-resident)."""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import regularizepsf_b200 as rp
from regularizepsf_b200 import _native
from regularizepsf_b200.device import DeviceCube

B = int(sys.argv[1]) if len(sys.argv) > 1 else 8
P = int(sys.argv[2]) if len(sys.argv) > 2 else 256
HW = int(sys.argv[3]) if len(sys.argv) > 3 else 2048
steps = 20
coords = [tuple(int(v) for v in c) for c in rp.calculate_covering((HW, HW), P)]
g = torch.Generator(device="cuda").manual_seed(1)
kernel = torch.randn((len(coords), P, P), dtype=torch.complex64, device="cuda", generator=g)
t = rp.ArrayPSFTransform(DeviceCube(coords, kernel))
frames = torch.rand((B, HW, HW), device="cuda", generator=g) * 1000
out = torch.empty_like(frames)
nt = t._native_transform("float32")
plan = nt.plan(HW, HW, 0, 0, HW, B)
lib = _native.load()
for _ in range(5):
    t._apply_device(frames, "float32", 0, out=out)
torch.cuda.synchronize()
lib.rpsf_plan_enable_timing(plan, 1)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(steps):
    t._apply_device(frames, "float32", 0, out=out)
e1.record()
torch.cuda.synchronize()
ms = (ctypes.c_double * 3)(); calls = ctypes.c_int()
lib.rpsf_plan_read_timing(plan, ms, ctypes.byref(calls))
per = [1e3 * ms[i] / calls.value / B for i in range(3)]
tot = 1e3 * e0.elapsed_time(e1) / steps / B
print(f"B={B} P={P} HW={HW}: us/frame total {tot:.1f}  k1 {per[0]:.1f}  k2 {per[1]:.1f}  k3 {per[2]:.1f}  "
      f"-> {HW * HW / tot:.0f} Mpix/s")
