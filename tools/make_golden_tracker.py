#!/usr/bin/env python
"""Golden fixtures for the tracker host loops (tests/golden/tracker_*.npz): the UNMODIFIED reference
``BaseTrackerPredictor.forward`` (vggsfm/models/track_modules/base_track_predictor.py:81-238) and ``refine_track`` /
``compute_score_fn`` (refine_track.py:24-294) run on CPU with their own CorrBlock / sample_features4d / embeddings; the
learned transformer is replaced on both sides by the deterministic stand-in tests/helpers.py:tiny_former (it is not on
the hot path and its weights would not fit a fixture), the fine feature net by one 3x3 convolution.  kornia is absent:
its two tiny functions used by compute_score_fn (create_meshgrid, dsnt.spatial_expectation2d) are restated here
[3P-memory].  The coarse feature maps are rounded to float16 before the run and stored as float16 (exact, and half the
size).  Needs a reference checkout:   VGGSFM_REFERENCE=/path/to/vggsfm python tools/make_golden_tracker.py"""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import reference_shim  # noqa: E402
from tests.helpers import tiny_former  # noqa: E402


def create_meshgrid(height, width, normalized_coordinates=True, device=None, dtype=torch.float32):
    xs = torch.linspace(-1, 1, width, device=device, dtype=dtype) if normalized_coordinates else torch.arange(width, device=device, dtype=dtype)
    ys = torch.linspace(-1, 1, height, device=device, dtype=dtype) if normalized_coordinates else torch.arange(height, device=device, dtype=dtype)
    gy, gx = torch.meshgrid(ys, xs, indexing="ij")
    return torch.stack([gx, gy], dim=-1)[None]


def spatial_expectation2d(inp, normalized_coordinates=True):
    B, N, H, W = inp.shape
    grid = create_meshgrid(H, W, normalized_coordinates, inp.device, inp.dtype)
    flat = inp.reshape(B, N, -1)
    ex = (grid[..., 0].reshape(-1) * flat).sum(-1, keepdim=True)
    ey = (grid[..., 1].reshape(-1) * flat).sum(-1, keepdim=True)
    return torch.cat([ex, ey], dim=-1)


def score_fn_inputs():
    """(B, N, S, query features, patch features, tracks) of the compute_score_fn cases: C = 8, 31x31 patches, sradius 2;
    some neighbourhoods get clamped at the patch border."""
    g = torch.Generator().manual_seed(0)
    out = []
    for B, N, S in ((1, 5, 4), (2, 3, 3)):
        qf = torch.randn(B, N, 8, generator=g)
        pf = torch.randn(B * N, S, 8, 31, 31, generator=g)
        trk = torch.rand(B * N, S, 1, 2, generator=g) * 34 - 2
        out.append((B, N, S, qf, pf, trk))
    return out


def state(m):
    return {k: v.detach().numpy() for k, v in m.state_dict().items()}


def main():
    reference_shim.install()
    from vggsfm.models.track_modules import base_track_predictor as bp
    from vggsfm.models.track_modules import refine_track as rt
    rt.create_meshgrid = create_meshgrid
    rt.dsnt = types.SimpleNamespace(spatial_expectation2d=spatial_expectation2d)
    cfg = types.SimpleNamespace(MODEL=types.SimpleNamespace(TRACK=types.SimpleNamespace(efficient_corr=False)))
    out = os.path.join(ROOT, "tests", "golden")
    with torch.no_grad():
        # ---- coarse-like predictor: stride 4, 5 levels, radius 3, 32 channels (transformer_dim 312 >= 311 inputs)
        torch.manual_seed(0)
        ref = bp.BaseTrackerPredictor(stride=4, corr_levels=5, corr_radius=3, latent_dim=32, hidden_size=16, use_spaceatt=False,
                                      depth=1, fine=False, cfg=cfg)
        ref.updateformer = tiny_former(ref.transformer_dim, 34, seed=1)
        ref.eval()
        # smooth feature maps (a coarse random field, bilinearly upsampled, + 5 % noise): the correlation landscape a
        # trained encoder produces, not white noise
        fmaps = torch.nn.functional.interpolate(torch.randn(10, 32, 5, 7), size=(32, 48), mode="bilinear", align_corners=True)
        fmaps = (fmaps + 0.05 * torch.randn_like(fmaps)).reshape(2, 5, 32, 32, 48).half().float()
        qp = torch.rand(2, 20, 2) * torch.tensor([48 * 4 - 8.0, 32 * 4 - 8.0]) + 4.0
        preds, vis, feats, qfeat = ref(qp, fmaps, iters=4, return_feat=True)
        np.savez_compressed(os.path.join(out, "tracker_coarse.npz"), fmaps=fmaps.half().numpy(), qp=qp.numpy(),
                            preds=torch.stack(preds).numpy(), vis=vis.numpy(), feats=feats.numpy(), qfeat=qfeat.numpy(),
                            transformer_dim=ref.transformer_dim,
                            **{"norm." + k: v for k, v in state(ref.norm).items()},
                            **{"ffeat." + k: v for k, v in state(ref.ffeat_updater).items()},
                            **{"vis." + k: v for k, v in state(ref.vis_predictor).items()})
        print("coarse", torch.stack(preds).shape, float(vis.mean()), ref.transformer_dim)
        # ---- fine stage: 31x31 patches, stride 1, one query per patch
        torch.manual_seed(1)
        fine = bp.BaseTrackerPredictor(stride=1, corr_levels=3, corr_radius=3, latent_dim=32, hidden_size=16, use_spaceatt=False,
                                       depth=1, fine=True, cfg=cfg)
        fine.updateformer = tiny_former(fine.transformer_dim, 34, seed=2)
        fine.eval()
        fnet = torch.nn.Conv2d(3, 32, 3, padding=1)
        images = torch.nn.functional.interpolate(torch.rand(4, 3, 9, 9), size=(72, 72), mode="bilinear", align_corners=True)[None]
        images = images + 0.02 * torch.rand_like(images)
        coarse = torch.rand(1, 4, 7, 2) * 60 + 6
        coarse[0, :, 0] = torch.tensor([1.3, 70.2])          # a track whose patch is clamped at the border
        tracks, score = rt.refine_track(images, fnet, fine, coarse, compute_score=True, pradius=15, sradius=2, fine_iters=3)
        np.savez_compressed(os.path.join(out, "tracker_fine.npz"), images=images.numpy(), coarse=coarse.numpy(),
                            tracks=tracks.numpy(), score=score.numpy(), transformer_dim=fine.transformer_dim,
                            **{"fnet." + k: v for k, v in state(fnet).items()},
                            **{"norm." + k: v for k, v in state(fine.norm).items()},
                            **{"ffeat." + k: v for k, v in state(fine.ffeat_updater).items()})
        print("fine", tracks.shape, score.shape, float(score.mean()), fine.transformer_dim)
        # ---- the two embeddings on their own
        from vggsfm.models.utils import get_2d_embedding, get_2d_sincos_pos_embed
        xy = torch.randn(3, 7, 2) * 5
        np.savez_compressed(os.path.join(out, "tracker_embed.npz"), xy=xy.numpy(), e16=get_2d_embedding(xy, 16, cat_coords=False).numpy(),
                            e64c=get_2d_embedding(xy, 64, cat_coords=True).numpy(),
                            pos216=get_2d_sincos_pos_embed(216, grid_size=(31, 31)).numpy(),
                            pos664=get_2d_sincos_pos_embed(664, grid_size=(6, 9)).numpy())
        # ---- compute_score_fn, including the reference's two indexing quirks (refine_track.py:256-276), on the seeded
        # inputs of score_fn_inputs(); the patch features are too large to store, a fixed sample of them pins the draw
        rec = {}
        for k, (B, N, S, qf, pf, trk) in enumerate(score_fn_inputs()):
            rec[f"score{k}"] = rt.compute_score_fn(qf, pf, trk, 2, 31, B, N, S, 8).numpy()
            rec[f"qf{k}"], rec[f"trk{k}"], rec[f"pf_sample{k}"] = qf.numpy(), trk.numpy(), pf.reshape(-1)[::97].numpy()
        np.savez_compressed(os.path.join(out, "tracker_score_fn.npz"), **rec)


if __name__ == "__main__":
    main()
