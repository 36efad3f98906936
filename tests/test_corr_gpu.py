"""GPU parity of the fused correlation+sampling kernel: reference goldens, the float32 torch oracle on
fresh inputs (float pyramid: 2e-4 of range; half pyramid as under the reference's fp16 autocast: 1e-2),
and linearity in the targets at the BASELINE C4 shape."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import corr_oracle as co

pytestmark = pytest.mark.gpu
GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "corr_*.npz")))


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_against_reference_golden(cuda_dev, path):
    from vggsfm_b200.corr import CorrBlock, EfficientCorrBlock
    g = np.load(path)
    # fmaps are stored as float16, exactly the values the reference ran on
    f, t, c = (torch.from_numpy(g[k].astype(np.float32)).to(cuda_dev) for k in ("fmaps", "targets", "coords"))
    L, r = int(g["num_levels"]), int(g["radius"])
    cb = CorrBlock(f, num_levels=L, radius=r, half=False)
    cb.corr(t)
    out = cb.sample(c).cpu().numpy()
    assert out.shape == g["out_zeros"].shape
    assert np.abs(out - g["out_zeros"]).max() < 2e-4 * np.abs(g["out_zeros"]).max()
    eb = EfficientCorrBlock(f, num_levels=L, radius=r, half=False)
    outb = eb.sample(c, t).cpu().numpy()
    assert np.abs(outb - g["out_border"]).max() < 2e-4 * np.abs(g["out_border"]).max()


@pytest.mark.parametrize("B,S,C,H,W,N,L,r", [(1, 4, 128, 64, 64, 50, 5, 4), (7, 3, 32, 31, 31, 1, 3, 3), (2, 2, 64, 24, 40, 9, 3, 4)])
def test_against_oracle_float_and_half(cuda_dev, B, S, C, H, W, N, L, r):
    from vggsfm_b200.corr import CorrBlock
    g = torch.Generator().manual_seed(B * 100 + S)
    f = torch.randn(B, S, C, H, W, generator=g)
    t = torch.randn(B, S, N, C, generator=g)
    c = torch.rand(B, S, N, 2, generator=g) * torch.tensor([W + 8.0, H + 8.0]) - 4.0     # crosses every border
    ref = co.corr_sample(f, t, c, L, r).numpy()
    rng = np.abs(ref).max()
    cb = CorrBlock(f.to(cuda_dev), num_levels=L, radius=r, half=False)
    cb.corr(t.to(cuda_dev))
    out = cb.sample(c.to(cuda_dev)).cpu().numpy()
    assert np.abs(out - ref).max() < 2e-4 * rng
    cbh = CorrBlock(f.to(cuda_dev), num_levels=L, radius=r, half=True)
    cbh.corr(t.to(cuda_dev))
    outh = cbh.sample(c.to(cuda_dev)).cpu().numpy()
    assert np.abs(outh - ref).max() < 1e-2 * rng


def test_c4_shape_linearity(cuda_dev):
    """BASELINE C4 coarse shape per chunk is [1,128,128,128,128] x 1024 queries; run 16 frames of it at full
    spatial size and check linearity in the targets and zero response far outside the map."""
    from vggsfm_b200.corr import CorrBlock
    g = torch.Generator().manual_seed(0)
    f = torch.randn(1, 16, 128, 128, 128, generator=g).to(cuda_dev)
    t1 = torch.randn(1, 16, 1024, 128, generator=g).to(cuda_dev)
    t2 = torch.randn(1, 16, 1024, 128, generator=g).to(cuda_dev)
    c = (torch.rand(1, 16, 1024, 2, generator=g) * 119 + 4).to(cuda_dev)
    cb = CorrBlock(f, num_levels=5, radius=4, half=False)
    outs = []
    for t in (t1, t2, t1 + 2 * t2):
        cb.corr(t)
        outs.append(cb.sample(c))
    assert outs[0].shape == (1, 16, 1024, 405)
    err = (outs[2] - (outs[0] + 2 * outs[1])).abs().max().item()
    assert err < 1e-3 * outs[2].abs().max().item()
    cb.corr(t1)
    far = cb.sample(torch.full_like(c, -1000.0))
    assert far.abs().max().item() == 0.0


@pytest.mark.parametrize("H,W,N,L,r", [(32, 32, 130, 3, 4), (24, 64, 256, 4, 3), (128, 128, 128, 5, 4)])
def test_tensor_core_path_matches_cuda_core_path(cuda_dev, H, W, N, L, r):
    """csrc/corr_tc.cu (tcgen05 kind::f16, footprint extraction from TMEM) against csrc/corr.cu on the same half
    pyramid: both round targets and features to fp16 and accumulate in fp32, only the summation order differs (1e-3 of
    the value range); queries on, near and beyond the border, a ragged last 128-query tile, non-square maps."""
    import torch
    from vggsfm_b200.corr import CorrBlock
    g = torch.Generator(device=cuda_dev).manual_seed(H + N)
    B, S, C = 1, 3, 128
    fm = torch.randn(B, S, C, H, W, device=cuda_dev, generator=g)
    tg = torch.randn(B, S, N, C, device=cuda_dev, generator=g)
    co = torch.rand(B, S, N, 2, device=cuda_dev, generator=g) * torch.tensor([W + 10.0, H + 10.0], device=cuda_dev) - 5.0
    co[0, 0, 0] = torch.tensor([0.0, 0.0], device=cuda_dev)
    co[0, 0, 1] = torch.tensor([W - 1.0, H - 1.0], device=cuda_dev)
    co[0, 1, 2] = torch.tensor([3.5, 7.25], device=cuda_dev)
    a = CorrBlock(fm, num_levels=L, radius=r, half=True, tc=True)
    assert a._pyr.tc_tiles is not None
    b = CorrBlock(fm, num_levels=L, radius=r, half=True, tc=False)
    assert b._pyr.tc_tiles is None
    a.corr(tg)
    b.corr(tg)
    ya, yb = a.sample(co), b.sample(co)
    torch.cuda.synchronize()
    scale = yb.abs().max().item()
    assert scale > 1.0
    assert (ya - yb).abs().max().item() <= 1e-3 * scale, (ya - yb).abs().max().item() / scale
