"""Golden fixtures for the correlation path from the UNMODIFIED reference CorrBlock / EfficientCorrBlock.  The feature
maps are rounded to float16 before the run and stored as float16 (exact, and half the size).  Needs a reference
checkout:  VGGSFM_REFERENCE=/path/to/vggsfm python tools/make_golden_corr.py"""
import os
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")
from oracle import reference_shim as rs   # noqa: E402

rs.install()
from vggsfm.models.track_modules.blocks import CorrBlock, EfficientCorrBlock   # noqa: E402

CASES = {
    # name: (B, S, C, H, W, N, levels, radius, coordinate range)
    "corr_coarse_small": (1, 2, 128, 32, 40, 24, 5, 4, (-6.0, 44.0)),     # 5 levels r=4 like the coarse tracker, borders hit
    "corr_fine_patch": (3, 2, 32, 31, 31, 1, 3, 3, (1.0, 29.0)),          # fine tracker: one query per 31x31 patch
}


def main():
    out_dir = os.path.join(ROOT, "tests", "golden")
    for name, (B, S, C, H, W, N, L, r, (lo, hi)) in CASES.items():
        g = torch.Generator().manual_seed(len(name))
        fmaps = torch.randn(B, S, C, H, W, generator=g).half().float()
        targets = torch.randn(B, S, N, C, generator=g)
        coords = torch.rand(B, S, N, 2, generator=g) * (hi - lo) + lo
        coords[0, 0, 0] = torch.tensor([3.0, 7.0])          # exactly integer coordinates
        cb = CorrBlock(fmaps, num_levels=L, radius=r)
        cb.corr(targets)
        out = cb.sample(coords)
        eb = EfficientCorrBlock(fmaps, num_levels=L, radius=r)
        out_b = eb.sample(coords, targets)
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), fmaps=fmaps.half().numpy(), targets=targets.numpy(), coords=coords.numpy(),
                            num_levels=L, radius=r, out_zeros=out.numpy(), out_border=out_b.numpy())
        print(name, out.shape, float(out.abs().mean()))


if __name__ == "__main__":
    main()
