"""CPU: the triangulation oracle (oracle/tri_oracle.py) against the committed golden fixtures produced by
the reference itself (tools/make_golden.py)."""
import glob
import os

import numpy as np
import pytest

from oracle import tri_oracle as to

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "tri_*.npz")))


def load(path):
    g = dict(np.load(path))
    g["extra"] = g["extra_params"] if g["extra_params"].shape[0] else None
    return g


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_matches_reference_golden(path):
    g = load(path)
    tn = to.cam_from_img(g["tracks"].astype(np.float64), g["intrinsics"], g["extra"])
    assert np.abs(tn - g["tn"]).max() < 1e-12          # same iteration, same global stop
    pts, num, mask = to.triangulate_tracks(g["extrinsics"], g["tn"], g["pairs"], g["vis"], g["score"])
    if bool(g["pinned"]):
        assert np.array_equal(num, g["inlier_num"])
        assert np.array_equal(mask, g["inlier_mask"])
        assert np.abs(pts - g["points"]).max() <= 1e-9 * np.abs(g["points"]).max()
    else:
        # reference run with its unstable sort: tie order may differ, the outcome must still agree
        same = (num == g["inlier_num"])
        assert same.mean() >= 0.95
        close = np.linalg.norm(pts - g["points"], axis=1) <= 1e-3
        assert close.mean() >= 0.95
    v, d = to.filter_all_points3D(g["points"], g["tracks"].astype(np.float64), g["extrinsics"], g["intrinsics"],
                                  g["extra"], max_reproj_error=1.0, return_detail=True)
    assert np.array_equal(v, g["filt_valid"]) and np.array_equal(d, g["filt_detail"])
    v2, _ = to.filter_all_points3D(g["points"], g["tracks"].astype(np.float64), g["extrinsics"], g["intrinsics"],
                                   g["extra"], max_reproj_error=4.0, check_triangle=False)
    assert np.array_equal(v2, g["filt_valid_notri"])
    p2d, pcam = to.project_3D_points(g["points"], g["extrinsics"], g["intrinsics"], g["extra"])
    assert np.abs(p2d - g["proj2d"]).max() < 1e-8 and np.abs(pcam - g["projcam"]).max() < 1e-10
    bp, bche, bang = to.triangulate_by_pair(g["extrinsics"], g["tn"])
    assert np.array_equal(bche, g["pair_cheirality"])
    assert np.nanmax(np.abs(bp - g["pair_points"]) / (1 + np.abs(g["pair_points"]))) < 1e-7
    assert np.nanmax(np.abs(bang - g["pair_angle"])) < 1e-7


def test_oracle_matches_live_reference():
    """The reference's triangulate_tracks run with its default arguments after torch.manual_seed(3) (stable sort),
    recorded by tools/make_golden.py: the oracle replays the same hypothesis draw and reaches the same result."""
    import torch
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "triangulate_tracks_10x40_radial.npz"))
    torch.manual_seed(3)
    pairs = to.draw_pairs(10, 256)
    po, no, mo = to.triangulate_tracks(g["extrinsics"], g["tn"], pairs, g["vis"], g["score"])
    assert np.array_equal(no, g["inlier_num"]) and np.array_equal(mo, g["inlier_mask"])
    assert np.abs(po - g["points"]).max() < 1e-9


def test_undistortion_quirk_is_reproduced():
    """SURVEY Appendix A.3: the reference's damped Newton stops ~4e-6 short of the true undistortion."""
    from vggsfm_b200.synthetic import make_scene
    sc = make_scene(4, 50, "SIMPLE_RADIAL", seed=5)
    k = sc.extra_params[:, 0]
    tn_d = (sc.tracks.astype(np.float64) - 512.0) / 1000.0
    und, iters = to.iterative_undistortion(k, tn_d)
    u, v = to.apply_distortion(k, und[..., 0], und[..., 1])
    err = np.abs(np.stack([u, v], -1) - tn_d).max()
    assert 2 <= iters < 100 and err < 1e-4
