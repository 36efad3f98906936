"""GPU parity of the tracker host loops (vggsfm_b200/tracker.py) on the CUDA correlation / sampling kernels against
goldens produced by the UNMODIFIED reference loops on CPU (tools/make_golden_tracker.py): BaseTrackerPredictor.forward
(base_track_predictor.py:81-238) and refine_track + compute_score_fn (refine_track.py:24-294).  Tolerances: the fused
kernel sums the 32-channel dot products in a different order than torch.matmul (float32); per-iteration bars in the
tests (the loop amplifies rounding differences, see the comment there)."""
import os
import types

import numpy as np
import pytest

from tests.helpers import tiny_former, to_dev

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _predictor(g, dev, stride, levels, radius, fine, former_seed):
    import torch
    import torch.nn as nn
    latent = 32
    p = types.SimpleNamespace(stride=stride, latent_dim=latent, corr_levels=levels, corr_radius=radius, fine=fine,
                              flows_emb_dim=latent // 2, transformer_dim=int(g["transformer_dim"]), efficient_corr=False)
    p.updateformer = tiny_former(p.transformer_dim, latent + 2, seed=former_seed).to(dev)
    p.norm = nn.GroupNorm(1, latent).to(dev)
    p.norm.load_state_dict({k[5:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("norm.")})
    p.ffeat_updater = nn.Sequential(nn.Linear(latent, latent), nn.GELU()).to(dev)
    p.ffeat_updater.load_state_dict({k[6:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("ffeat.")})
    if not fine:
        p.vis_predictor = nn.Sequential(nn.Linear(latent, 1)).to(dev)
        p.vis_predictor.load_state_dict({k[4:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("vis.")})
    return p


def test_track_predictor_forward_matches_reference(cuda_dev):
    import torch
    from vggsfm_b200 import tracker as tk
    g = np.load(os.path.join(GOLD, "tracker_coarse.npz"))
    p = _predictor(g, cuda_dev, 4, 5, 3, False, 1)
    fmaps = to_dev(g["fmaps"].astype(np.float32), cuda_dev)            # stored as float16, exactly what the reference ran on
    preds, vis, feats, qfeat = tk.track_predictor_forward(p, to_dev(g["qp"], cuda_dev), fmaps, iters=4,
                                                         return_feat=True)
    assert len(preds) == 4
    got = torch.stack(preds).cpu().numpy()
    assert got.shape == g["preds"].shape
    # The loop feeds its own output back through ~250 correlation samples per token: one float32 ulp of the coordinates
    # (1.5e-5 px at x ~ 190) grows 3-13x per iteration between ANY two correct implementations (the CPU emulation with
    # oracle/corr_oracle.py shows 1.5e-5 / 2e-4 / 7e-4 / 2e-3 px against these goldens).  A wrong axis order, embedding or
    # update rule moves the 0.3 px per-iteration steps themselves and fails the first bars by two orders of magnitude.
    for it, tol in enumerate((1e-3, 3e-3, 1e-2, 3e-2)):
        d = np.abs(got[it] - g["preds"][it]).max()
        assert d < tol, (it, d)
    assert np.abs(got[0] - g["qp"][:, None]).max() > 0.05            # the predictor does move the tracks
    assert np.abs(vis.cpu().numpy() - g["vis"]).max() < 1e-2
    assert np.abs(feats.cpu().numpy() - g["feats"]).max() < 3e-2
    assert np.abs(qfeat.cpu().numpy() - g["qfeat"]).max() < 1e-5
    # frame 0 stays the query (base_track_predictor.py:219)
    assert np.array_equal(got[-1][:, 0], got[0][:, 0])


def test_refine_track_matches_reference(cuda_dev):
    import torch
    import torch.nn as nn
    from vggsfm_b200 import tracker as tk
    g = np.load(os.path.join(GOLD, "tracker_fine.npz"))
    fine = _predictor(g, cuda_dev, 1, 3, 3, True, 2)
    fnet = nn.Conv2d(3, 32, 3, padding=1).to(cuda_dev)
    fnet.load_state_dict({k[5:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("fnet.")})
    tracks, score = tk.refine_track(to_dev(g["images"], cuda_dev), fnet, fine, to_dev(g["coarse"], cuda_dev), compute_score=True,
                                    pradius=15, sradius=2, fine_iters=3)
    assert np.abs(tracks.cpu().numpy() - g["tracks"]).max() < 2e-3, np.abs(tracks.cpu().numpy() - g["tracks"]).max()
    assert np.abs(score.cpu().numpy() - g["score"]).max() < 1e-3
    assert np.array_equal(tracks.cpu().numpy()[:, 0], g["coarse"][:, 0])            # query frame untouched
