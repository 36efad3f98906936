"""Accuracy / timing check of the tcgen05 INT8 (Ozaki) SYRK against numpy float64.
   python tools/syrk_i8_check.py [Dpad Kpad slices]"""
import ctypes
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vggsfm_b200 import _lib       # noqa: E402

dev = torch.device("cuda:0")
if len(sys.argv) > 1 and sys.argv[1] == "rate":
    L = _lib.lib()
    torch.zeros(1, device=dev)
    for mode, name in [(0, "SW64  N=128"), (1, "SW64  N=256"), (2, "SW128 N=128"), (3, "SW128 N=256"), (4, "none  N=128"), (5, "none  N=256"),
                       (8, "SW64  N=128 A-in-TMEM"), (9, "SW64  N=256 A-in-TMEM")]:
        c = ctypes.c_double()
        _lib.check(L.vgg_syrk_ozaki_mma_rate(4096, mode, ctypes.byref(c), None), "rate")
        n = 256 if mode & 1 else 128
        print(f"kind::i8 M=128 {name} K=32: {c.value:7.1f} cycles/MMA -> {128 * n * 32 / c.value:7.0f} MAC/clk/SM")
    sys.exit(0)
Dpad = int(sys.argv[1]) if len(sys.argv) > 1 else 256
Kpad = int(sys.argv[2]) if len(sys.argv) > 2 else 640
s = int(sys.argv[3]) if len(sys.argv) > 3 else 7
L = _lib.lib()
rng = np.random.default_rng(0)
Z = rng.normal(size=(Kpad, Dpad)) * np.exp(rng.uniform(-6, 6, size=(1, Dpad)))     # column scales over 5 decades
Z[:, -3:] = 0.0                                                                     # padding columns
Z[rng.uniform(size=Z.shape) < 0.3] = 0.0
Zt = torch.from_numpy(Z).to(dev)
C = torch.zeros(Dpad, Dpad, dtype=torch.float64, device=dev)
nb = ctypes.c_size_t()
_lib.check(L.vgg_syrk_ozaki_workspace_bytes(Kpad, Dpad, s, ctypes.byref(nb)), "ws")
ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
st = torch.cuda.current_stream().cuda_stream
_lib.check(L.vgg_syrk_ozaki(Kpad, Dpad, Zt.data_ptr(), C.data_ptr(), s, ws.data_ptr(), ws.numel(), st), "syrk")
torch.cuda.synchronize()
got = np.tril(C.cpu().numpy())                      # the kernel writes the row-major LOWER triangle
upper_untouched = not np.triu(C.cpu().numpy(), 1).any()
got = got + np.tril(got, -1).T
ref = -(Z.T @ Z)
bound = np.abs(Z).T @ np.abs(Z) + 1e-300
err = np.abs(got - ref) / bound
print(f"Dpad={Dpad} Kpad={Kpad} slices={s}: max |err| / (|Z|^T|Z|) = {err.max():.3e}   symmetric: {upper_untouched}  "
      f"nonzero frac {np.mean(got != 0):.3f}")
if err.max() > 1e-6:
    i, j = np.unravel_index(np.argmax(err), err.shape)
    print("worst at", i, j, got[i, j], ref[i, j])
    bad = err > 1e-6
    print("bad rows (first 16):", np.nonzero(bad.any(1))[0][:16], "bad cols:", np.nonzero(bad.any(0))[0][:16], "count", int(bad.sum()))
    blk = bad.reshape(Dpad // 128, 128, Dpad // 128, 128).any(axis=(1, 3))
    print("bad 128-blocks:\n", blk.astype(int))
    print("got[0,:4]", got[0, :4], "ref[0,:4]", ref[0, :4], "ratio", got[0, :4] / ref[0, :4])
if len(sys.argv) > 4:
    reps = 10
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        L.vgg_syrk_ozaki(Kpad, Dpad, Zt.data_ptr(), C.data_ptr(), s, ws.data_ptr(), ws.numel(), st)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        L.vgg_syrk_ozaki(Kpad, Dpad, Zt.data_ptr(), C.data_ptr(), s, ws.data_ptr(), ws.numel(), st)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    flop = 2.0 * Kpad * Dpad * (Dpad + 128) / 2
    print(f"  {ms:.3f} ms per call (rowmax + slice + SYRK)  = {flop / ms / 1e9:.1f} TFLOP/s FP64-equivalent")
