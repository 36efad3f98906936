#!/usr/bin/env python
"""Golden fixtures for the tensor <-> scene-object marshalling rules (tests/golden/marshal_*.npz).

Runs the UNMODIFIED reference loop ``batch_matrix_to_pycolmap`` (vggsfm/utils/tensor_to_pycolmap.py:16-160) and its
inverse ``pycolmap_to_batch_matrix`` (:163-214) with ``vggsfm_b200.reconstruction`` standing in for the absent
``pycolmap`` module -- i.e. the reference's own O(S*P) Python loops decide ids, point2D order, the 3000 clamp and the
camera sharing, and only the passive container classes are ours.  The flattened result is what
``Reconstruction.from_batch_matrix`` (the vectorised product path) must reproduce exactly.  Also pins the pure-torch
``get_valid_frame_mask`` (vggsfm/utils/triangulation.py:1222-1242), and records how the reference's COLMAP reader
(vggsfm/datasets/imc_helper.py:127-466) parses the binary model this package writes.  Needs a reference checkout:

    VGGSFM_REFERENCE=/path/to/vggsfm python tools/make_golden_marshal.py
"""
import os
import sys
import tempfile
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import reference_shim  # noqa: E402


def cases():
    from vggsfm_b200.synthetic import make_scene
    out = []
    for name, S, P, cam, shared in [("a", 5, 40, "SIMPLE_PINHOLE", False), ("b", 7, 33, "SIMPLE_RADIAL", True),
                                    ("c", 4, 25, "SIMPLE_RADIAL", False)]:
        sc = make_scene(S, P, cam, seed=len(name) + S, invisible_frac=0.35)
        masks = sc.mask.copy()
        masks[:, 3] = False              # no observations
        masks[1:, 6] = False             # one observation: not a point
        pts = sc.points3d.copy()
        pts[8] = [3500.0, 0.1, 2.0]      # beyond max_points3D_val: point exists, gets no observations (:131-133)
        pts[9] = [-3500.0, 0.1, 2.0]     # the clamp is one-sided (xyz < 3000): this one keeps its observations
        out.append(dict(name=name, cam=cam, shared=shared, pts=pts, extr=sc.extrinsics, K=sc.intrinsics,
                        extra=sc.extra_params, tracks=sc.tracks, masks=masks, size=np.array([1024, 768])))
    return out


def flatten(model):
    """model dict (Reconstruction.to_model()) -> flat arrays."""
    o = {}
    cids = sorted(model["cameras"])
    o["cam_ids"] = np.array(cids)
    o["cam_params"] = np.stack([np.pad(model["cameras"][c]["params"], (0, 4 - len(model["cameras"][c]["params"]))) for c in cids])
    o["cam_wh"] = np.array([[model["cameras"][c]["width"], model["cameras"][c]["height"]] for c in cids])
    iids = sorted(model["images"])
    o["img_ids"] = np.array(iids)
    o["img_cam"] = np.array([model["images"][i]["camera_id"] for i in iids])
    o["img_tvec"] = np.stack([model["images"][i]["tvec"] for i in iids])
    o["img_npts"] = np.array([len(model["images"][i]["point3D_ids"]) for i in iids])
    o["img_xys"] = np.concatenate([model["images"][i]["xys"].reshape(-1, 2) for i in iids])
    o["img_p3d"] = np.concatenate([np.asarray(model["images"][i]["point3D_ids"]).reshape(-1) for i in iids])
    pids = sorted(model["points3D"])
    o["pt_ids"] = np.array(pids)
    o["pt_xyz"] = np.stack([model["points3D"][p]["xyz"] for p in pids])
    o["pt_tracklen"] = np.array([len(model["points3D"][p]["track"]) for p in pids])
    o["pt_track"] = np.concatenate([np.asarray(model["points3D"][p]["track"], dtype=np.int64).reshape(-1, 2) for p in pids])
    return o


def read_back(path):
    """The reference reader's view of the binary model under ``path`` -> flat arrays (the .bin bytes it parsed included)."""
    sys.modules.setdefault("h5py", types.ModuleType("h5py"))          # imported at module scope there, unused by the readers
    from vggsfm.datasets import imc_helper as ih
    cams, ims, pts = ih.read_model(path, ext=".bin")
    o = {}
    for f in ("cameras", "images", "points3D"):
        with open(os.path.join(path, f + ".bin"), "rb") as fh:
            o["bin_" + f] = np.frombuffer(fh.read(), dtype=np.uint8)
    cids, iids, pids = sorted(cams), sorted(ims), sorted(pts)
    o["cam_ids"] = np.array(cids)
    o["cam_model"] = np.array([cams[c].model for c in cids])
    o["cam_wh"] = np.array([[cams[c].width, cams[c].height] for c in cids])
    o["cam_params"] = np.stack([cams[c].params for c in cids])
    o["img_ids"] = np.array(iids)
    o["img_name"] = np.array([ims[i].name for i in iids])
    o["img_cam"] = np.array([ims[i].camera_id for i in iids])
    o["img_R"] = np.stack([ims[i].qvec2rotmat() for i in iids])
    o["img_tvec"] = np.stack([ims[i].tvec for i in iids])
    o["img_npts"] = np.array([len(ims[i].point3D_ids) for i in iids])
    o["img_xys"] = np.concatenate([ims[i].xys.reshape(-1, 2) for i in iids])
    o["img_p3d"] = np.concatenate([ims[i].point3D_ids.reshape(-1) for i in iids])
    o["pt_ids"] = np.array(pids)
    o["pt_xyz"] = np.stack([pts[p].xyz for p in pids])
    o["pt_rgb"] = np.stack([pts[p].rgb for p in pids])
    o["pt_tracklen"] = np.array([len(pts[p].image_ids) for p in pids])
    o["pt_track"] = np.concatenate([np.stack([pts[p].image_ids, pts[p].point2D_idxs], 1).reshape(-1, 2) for p in pids])
    return o


def main():
    reference_shim.install()
    import vggsfm_b200.reconstruction as rc
    sys.modules["pycolmap"] = rc                   # the reference's loops build OUR passive containers
    from vggsfm.utils import tensor_to_pycolmap as t2p
    t2p.pycolmap = rc
    from vggsfm.utils.triangulation import get_valid_frame_mask
    t = torch.from_numpy
    for c in cases():
        rec = t2p.batch_matrix_to_pycolmap(t(c["pts"]), t(c["extr"]), t(c["K"]), t(c["tracks"]), t(c["masks"]), t(c["size"]),
                                           shared_camera=c["shared"], camera_type=c["cam"],
                                           extra_params=t(c["extra"]) if c["extra"] is not None else None)
        flat = flatten(rec.to_model())
        back = t2p.pycolmap_to_batch_matrix(rec, device="cpu", camera_type=c["cam"])
        flat["back_pts"], flat["back_extr"], flat["back_K"] = back[0].numpy(), back[1].numpy(), back[2].numpy()
        if back[3] is not None:
            flat["back_extra"] = back[3].numpy()
        np.savez_compressed(os.path.join(ROOT, "tests", "golden", f"marshal_{c['name']}.npz"), **flat)
        print("marshal", c["name"], {k: v.shape for k, v in flat.items()})
    # get_valid_frame_mask
    g = torch.Generator().manual_seed(0)
    K = torch.zeros(12, 3, 3, dtype=torch.float64)
    K[:, 0, 0] = torch.tensor([50.0, 102.4, 102.3, 1000, 30720, 30721, 1000, 1000, 1000, 1000, -5, 1000])
    E = torch.randn(12, 3, 4, generator=g, dtype=torch.float64)
    E[6, 1, 3] = 30.0
    E[7, 2, 3] = -30.001
    ex = torch.zeros(12, 1, dtype=torch.float64)
    ex[8, 0] = 1.0
    ex[9, 0] = -1.0001
    m1 = get_valid_frame_mask(K, E, ex, 1024)
    m2 = get_valid_frame_mask(K, E, None, 1024)
    m3 = get_valid_frame_mask(K, E, ex[:, 0], 1024)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "valid_frame_mask.npz"), K=K.numpy(), E=E.numpy(), ex=ex.numpy(),
                        m1=m1.numpy(), m2=m2.numpy(), m3=m3.numpy())
    print("valid_frame_mask", m1.tolist())
    # case c built by this package's vectorised path, written as COLMAP binaries, parsed by the reference's reader
    c = cases()[2]
    rec = rc.batch_matrix_to_pycolmap(t(c["pts"]), t(c["extr"]), t(c["K"]), t(c["tracks"]), t(c["masks"]), t(c["size"]),
                                      shared_camera=c["shared"], camera_type=c["cam"], extra_params=t(c["extra"]))
    rec.set_point_colors(np.linspace(0, 1, rec.num_points3D())[:, None].repeat(3, 1))
    with tempfile.TemporaryDirectory() as d:
        rec.write(d)
        back = read_back(d)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "marshal_c_reader.npz"), **back)
    print("marshal_c_reader", {k: v.shape for k, v in back.items()})


if __name__ == "__main__":
    main()
