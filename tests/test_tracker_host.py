"""Host-side pieces of the tracker loops (vggsfm_b200/tracker.py) that run without a GPU: the two embeddings against
goldens produced by the reference (tools/make_golden_tracker.py), and compute_score_fn / the patch gather against the
reference's output recorded there."""
import os

import numpy as np
import torch

from tools.make_golden_tracker import score_fn_inputs
from vggsfm_b200 import tracker as tk

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_embeddings_match_reference_goldens():
    g = np.load(os.path.join(GOLD, "tracker_embed.npz"))
    xy = torch.from_numpy(g["xy"])
    assert np.abs(tk.get_2d_embedding(xy, 16, cat_coords=False).numpy() - g["e16"]).max() < 1e-6
    assert np.abs(tk.get_2d_embedding(xy, 64, cat_coords=True).numpy() - g["e64c"]).max() < 1e-6
    assert np.abs(tk.get_2d_sincos_pos_embed(216, (31, 31)).numpy() - g["pos216"]).max() < 1e-6
    assert np.abs(tk.get_2d_sincos_pos_embed(664, (6, 9)).numpy() - g["pos664"]).max() < 1e-6


def test_compute_score_fn_equals_live_reference():
    """Including the reference's two indexing quirks (refine_track.py:256-276), which a drop-in has to reproduce; the
    reference's output on the same seeded inputs is tests/golden/tracker_score_fn.npz."""
    g = np.load(os.path.join(GOLD, "tracker_score_fn.npz"))
    for k, (B, N, S, qf, pf, trk) in enumerate(score_fn_inputs()):
        # the inputs are drawn here again: they must be the ones the reference saw
        assert np.array_equal(qf.numpy(), g[f"qf{k}"]) and np.array_equal(trk.numpy(), g[f"trk{k}"])
        assert np.array_equal(pf.reshape(-1)[::97].numpy(), g[f"pf_sample{k}"])
        ref = g[f"score{k}"]
        got = tk.compute_score_fn(qf, pf, trk, 2, 31, B, N, S, 8)
        assert got.shape == ref.shape == (B, S, N)
        assert np.abs(got.numpy() - ref).max() < 1e-6
