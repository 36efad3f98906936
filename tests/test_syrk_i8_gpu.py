"""tcgen05 INT8 (Ozaki) SYRK (csrc/syrk_i8.cu, vgg_syrk_ozaki) against numpy float64: the error of every entry is
bounded relative to (|Z|^T |Z|)_ij -- the quantity a float64 dot product's own rounding error is bounded by --
at 2^-44 for 7 slices; fewer slices lose 8 bits each.  The LM solve, which runs this SYRK with 7 slices, is covered by
tests/test_ba_gpu.py."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _run(Z, s, dev):
    import torch
    from vggsfm_b200 import _lib
    L = _lib.lib()
    Kpad, Dpad = Z.shape
    Zt = torch.from_numpy(Z).to(dev)
    C = torch.zeros(Dpad, Dpad, dtype=torch.float64, device=dev)
    nb = ctypes.c_size_t()
    _lib.check(L.vgg_syrk_ozaki_workspace_bytes(Kpad, Dpad, s, ctypes.byref(nb)), "vgg_syrk_ozaki_workspace_bytes")
    ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.vgg_syrk_ozaki(Kpad, Dpad, Zt.data_ptr(), C.data_ptr(), s, ws.data_ptr(), ws.numel(),
                                    torch.cuda.current_stream().cuda_stream), "vgg_syrk_ozaki")
        torch.cuda.synchronize()
    full = C.cpu().numpy()
    assert not np.triu(full, 1).any()                  # only the row-major LOWER triangle is written (csrc/chol.cu factors it)
    low = np.tril(full)
    return low + np.tril(low, -1).T


def _case(Dpad, Kpad, seed):
    rng = np.random.default_rng(seed)
    Z = rng.normal(size=(Kpad, Dpad)) * np.exp(rng.uniform(-6, 6, size=(1, Dpad)))
    Z[rng.uniform(size=Z.shape) < 0.3] = 0.0
    Z[:, -5:] = 0.0
    return Z


@pytest.mark.parametrize("Dpad,Kpad,s,tol", [(128, 64, 7, 2.0 ** -44), (384, 1040, 7, 2.0 ** -44), (256, 640, 5, 2.0 ** -28),
                                             (256, 4096 + 16, 6, 2.0 ** -36), (640, 2000, 3, 2.0 ** -12)])
def test_matches_float64(cuda_dev, Dpad, Kpad, s, tol):
    Z = _case(Dpad, Kpad, Dpad + s)
    got = _run(Z, s, cuda_dev)
    ref = -(Z.T @ Z)
    bound = np.abs(Z).T @ np.abs(Z)
    err = np.abs(got - ref)
    assert np.all(err <= tol * bound + 1e-300), (err / (bound + 1e-300)).max()
    assert not got[:, -5:].any()


def test_accumulates_and_flags_nonfinite(cuda_dev):
    import torch
    Z = _case(256, 256, 1)
    got1 = _run(Z, 7, cuda_dev)
    assert np.abs(got1).max() > 0
    Z[17, 40] = np.nan
    got = _run(Z, 7, cuda_dev)
    assert np.isnan(got[40, :250]).all() and np.isnan(got[:250, 40]).all()
    ok = np.ones(256, bool)
    ok[40] = False
    assert np.isfinite(got[np.ix_(ok, ok)]).all()


def test_band_hint_skips_only_zero_blocks(cuda_dev):
    """With the band hint installed (k-block range per 128-column row block outside which Zt is zero) the kernel skips
    tiles whose ranges do not meet and shortens the rest: the result must equal the dense product of the same Z."""
    from vggsfm_b200 import _lib
    L = _lib.lib()
    Dpad, KB = 1024, 24
    Z = _case(Dpad, KB * 64, 11)
    nb = Dpad // 128
    rg = np.zeros((nb, 2), dtype=np.int32)
    for rb in range(nb):
        lo, hi = (0, KB) if rb == nb - 1 else (2 * rb, min(KB, 2 * rb + 7))        # last block: dense (the shared camera's column)
        rg[rb] = (lo, hi)
        Z[:lo * 64, rb * 128:(rb + 1) * 128] = 0.0
        Z[hi * 64:, rb * 128:(rb + 1) * 128] = 0.0
    ref = -(Z.T @ Z)
    bound = np.abs(Z).T @ np.abs(Z)
    dense = _run(Z, 7, cuda_dev)
    _lib.check(L.vgg_dev_set_syrk_ranges(rg.ctypes.data, rg.size), "ranges")
    try:
        got = _run(Z, 7, cuda_dev)
    finally:
        L.vgg_dev_set_syrk_ranges(None, 0)
    for name, m in (("dense", dense), ("band", got)):
        err = np.abs(m - ref)
        assert np.all(err <= 2.0 ** -44 * bound + 1e-300), (name, (err / (bound + 1e-300)).max())
    again = _run(Z, 7, cuda_dev)                       # and the plan goes back to dense when the hint is gone
    assert np.all(np.abs(again - ref) <= 2.0 ** -44 * bound + 1e-300)
