"""CPU: correlation oracle vs the goldens produced by the reference CorrBlock / EfficientCorrBlock."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import corr_oracle as co

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "corr_*.npz")))


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_corr_oracle_matches_reference_golden(path):
    g = np.load(path)
    # fmaps are stored as float16, exactly the values the reference ran on
    f, t, c = (torch.from_numpy(g[k].astype(np.float32)) for k in ("fmaps", "targets", "coords"))
    L, r = int(g["num_levels"]), int(g["radius"])
    out = co.corr_sample(f, t, c, L, r, border=False).numpy()
    # float32 volume + float32 normalise/unnormalise round trip in grid_sample: 1e-4 of the value range
    tol = 2e-4 * np.abs(g["out_zeros"]).max()
    assert np.abs(out - g["out_zeros"]).max() < tol
    outb = co.corr_sample(f, t, c, L, r, border=True).numpy()
    assert np.abs(outb - g["out_border"]).max() < 2e-4 * np.abs(g["out_border"]).max()
