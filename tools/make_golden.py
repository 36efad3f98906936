"""Generate tests/golden/tri_*.npz and triangulate_tracks_10x40_radial.npz by running the UNMODIFIED reference
(imported with stub third-party modules) on seeded synthetic inputs.  Needs a reference checkout:

    VGGSFM_REFERENCE=/path/to/vggsfm python tools/make_golden.py

Pinned cases run the reference with torch.sort forced stable (its unstable descending sort leaves the
order of equal inlier counts implementation-defined, see oracle/tri_oracle.py); the `unpinned` case runs
it exactly as shipped.  The hypothesis frame pairs are recorded by replaying the CPU RNG draw of
vggsfm/utils/triangulation.py:811-813 from the same seed.
"""
import os
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")

from oracle import reference_shim as rs          # noqa: E402
from oracle import tri_oracle as to              # noqa: E402
from vggsfm_b200.synthetic import make_scene     # noqa: E402

rs.install()
from vggsfm.utils import triangulation as rt               # noqa: E402
from vggsfm.utils import triangulation_helpers as rh       # noqa: E402

CASES = {
    # name: (S, N, camera, scene kwargs, max_ransac_iters, pinned)
    "tri_c1_8x256_pinhole": (8, 256, "SIMPLE_PINHOLE", dict(seed=0), 256, True),
    "tri_12x96_radial_outliers": (12, 96, "SIMPLE_RADIAL", dict(seed=1, invisible_frac=0.3, outlier_frac=0.1), 256, True),
    "tri_30x64_pinhole_256of435": (30, 64, "SIMPLE_PINHOLE", dict(seed=2, invisible_frac=0.2, outlier_frac=0.05), 256, True),
    "tri_40x48_radial_128hyp": (40, 48, "SIMPLE_RADIAL", dict(seed=3, invisible_frac=0.25, outlier_frac=0.08), 128, True),
    "tri_30x64_unpinned": (30, 64, "SIMPLE_PINHOLE", dict(seed=2, invisible_frac=0.2, outlier_frac=0.05), 256, False),
}

_sort = torch.sort


def _stable_sort(*a, **k):
    k["stable"] = True
    return _sort(*a, **k)


def main():
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    for name, (S, N, cam, kw, iters, pinned) in CASES.items():
        sc = make_scene(S, N, cam, **kw)
        K = torch.from_numpy(sc.intrinsics)
        E = torch.from_numpy(sc.extrinsics)
        ex = torch.from_numpy(sc.extra_params) if sc.extra_params is not None else None
        tracks = torch.from_numpy(sc.tracks)
        tn = rh.cam_from_img(tracks, K, ex)
        seed = 1234 + S
        torch.manual_seed(seed)
        pairs = to.draw_pairs(S, iters)
        torch.manual_seed(seed)
        if pinned:
            torch.sort = _stable_sort
        try:
            p, n, m = rt.triangulate_tracks(E, rs.contiguous_tracks(tn), max_ransac_iters=iters,
                                            track_vis=torch.from_numpy(sc.vis), track_score=torch.from_numpy(sc.score))
        finally:
            torch.sort = _sort
        v, d = rh.filter_all_points3D(p, tracks.double(), E, K, ex, max_reproj_error=1.0, return_detail=True)
        v2, _ = rh.filter_all_points3D(p, tracks.double(), E, K, ex, max_reproj_error=4.0, check_triangle=False)
        p2d, pcam = rh.project_3D_points(p, E, K, ex, return_points_cam=True)
        bp, bche, bang = rt.triangulate_by_pair(E[None], tn[None])
        np.savez_compressed(
            os.path.join(out_dir, name + ".npz"),
            extrinsics=sc.extrinsics, intrinsics=sc.intrinsics,
            extra_params=sc.extra_params if sc.extra_params is not None else np.zeros((0, 1)),
            tracks=sc.tracks, vis=sc.vis, score=sc.score, pairs=pairs.astype(np.int32), max_ransac_iters=iters,
            pinned=pinned, tn=tn.numpy(), points=p.numpy(), inlier_num=n.numpy(), inlier_mask=m.numpy(),
            filt_valid=v.numpy(), filt_detail=d.numpy(), filt_valid_notri=v2.numpy(), proj2d=p2d.numpy(),
            projcam=pcam.numpy(), pair_points=bp.numpy(), pair_cheirality=bche.numpy(), pair_angle=bang.numpy())
        print(name, "inliers/track mean", n.float().mean().item(), "valid", int(v.sum()))
    # triangulate_tracks alone on a radial scene with outliers, stable sort, default arguments (256 hypotheses)
    sc = make_scene(10, 40, "SIMPLE_RADIAL", seed=21, invisible_frac=0.2, outlier_frac=0.1)
    tn = rh.cam_from_img(torch.from_numpy(sc.tracks), torch.from_numpy(sc.intrinsics), torch.from_numpy(sc.extra_params))
    torch.manual_seed(3)
    torch.sort = _stable_sort
    try:
        p, n, m = rt.triangulate_tracks(torch.from_numpy(sc.extrinsics), rs.contiguous_tracks(tn),
                                        track_vis=torch.from_numpy(sc.vis), track_score=torch.from_numpy(sc.score))
    finally:
        torch.sort = _sort
    np.savez_compressed(os.path.join(out_dir, "triangulate_tracks_10x40_radial.npz"), extrinsics=sc.extrinsics,
                        tn=tn.numpy(), vis=sc.vis, score=sc.score, points=p.numpy(), inlier_num=n.numpy(),
                        inlier_mask=m.numpy())
    print("triangulate_tracks_10x40_radial", "inliers/track mean", n.float().mean().item())


if __name__ == "__main__":
    main()
