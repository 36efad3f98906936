"""The pycolmap-shaped scene object (vggsfm_b200/reconstruction.py) and the reference-held host rules around BA.

Pinned to the reference: tests/golden/marshal_*.npz were produced by the UNMODIFIED ``batch_matrix_to_pycolmap`` /
``pycolmap_to_batch_matrix`` loops (vggsfm/utils/tensor_to_pycolmap.py:16-214) and ``get_valid_frame_mask``
(vggsfm/utils/triangulation.py:1222-1242), see tools/make_golden_marshal.py; the vectorised product path must
reproduce them exactly.  The COLMAP binary files written here are the ones the reference's own reader
(vggsfm/datasets/imc_helper.py:127-466) parsed into tests/golden/marshal_c_reader.npz.  CPU only."""
import os

import numpy as np
import pytest
import torch

from tools.make_golden_marshal import cases, flatten
from vggsfm_b200 import colmap_io as cio
from vggsfm_b200 import reconstruction as rc

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
t = torch.from_numpy


def _build(c):
    return rc.batch_matrix_to_pycolmap(t(c["pts"]), t(c["extr"]), t(c["K"]), t(c["tracks"]), t(c["masks"]), t(c["size"]),
                                       shared_camera=c["shared"], camera_type=c["cam"],
                                       extra_params=t(c["extra"]) if c["extra"] is not None else None)


@pytest.mark.parametrize("idx", [0, 1, 2])
def test_from_batch_matrix_equals_reference_loop(idx):
    c = cases()[idx]
    g = np.load(os.path.join(GOLD, f"marshal_{c['name']}.npz"))
    rec = _build(c)
    assert rec._pending is not None                      # still lazy: no object graph was built to get here
    flat = flatten(rec.to_model())
    for k, v in flat.items():
        assert np.array_equal(v, g[k]), k
    back = rc.pycolmap_to_batch_matrix(rec, device="cpu", camera_type=c["cam"])
    assert np.array_equal(back[0].numpy(), g["back_pts"]) and np.array_equal(back[1].numpy(), g["back_extr"])
    assert np.array_equal(back[2].numpy(), g["back_K"])
    assert (back[3] is None) == ("back_extra" not in g.files)
    if back[3] is not None:
        assert np.array_equal(back[3].numpy(), g["back_extra"])
    # the rules themselves, stated once: ids 1..P' over >=2-inlier tracks; one-sided 3000 clamp drops observations only
    valid = np.nonzero(c["masks"].sum(0) >= 2)[0]
    assert list(flat["pt_ids"]) == list(range(1, len(valid) + 1))
    pid8 = int(np.nonzero(valid == 8)[0][0]) + 1
    pid9 = int(np.nonzero(valid == 9)[0][0]) + 1
    assert rec.points3D[pid8].track.length() == 0 and rec.points3D[pid9].track.length() == int(c["masks"][:, 9].sum())


@pytest.mark.parametrize("idx", [0, 1])
def test_live_reference_loop(idx):
    """The scene the reference's own loops built (our module standing in for pycolmap's containers), as recorded in
    tests/golden/marshal_*.npz by tools/make_golden_marshal.py, equals the vectorised build."""
    c = cases()[idx]
    a = np.load(os.path.join(GOLD, f"marshal_{c['name']}.npz"))
    b = flatten(_build(c).to_model())
    assert sorted(b) == sorted(k for k in a.files if not k.startswith("back_"))
    assert all(np.array_equal(a[k], b[k]) for k in b)


def test_get_valid_frame_mask_golden():
    from vggsfm_b200.bundle_adjustment import get_valid_frame_mask
    g = np.load(os.path.join(GOLD, "valid_frame_mask.npz"))
    K, E, ex = t(g["K"]), t(g["E"]), t(g["ex"])
    assert np.array_equal(get_valid_frame_mask(K, E, ex, 1024).numpy(), g["m1"])
    assert np.array_equal(get_valid_frame_mask(K, E, None, 1024).numpy(), g["m2"])
    assert np.array_equal(get_valid_frame_mask(K, E, ex[:, 0], 1024).numpy(), g["m3"])


def test_prepare_ba_options_rule():
    """triangulation_helpers.py:626-635: the three tolerances x10 (a zero default stays zero), 50 iterations."""
    from vggsfm_b200 import bundle_adjustment as ba
    d, o = ba.default_options(), ba.prepare_ba_options()
    assert o.max_num_iterations == 50 and d.max_num_iterations == 100
    assert o.function_tolerance == 10 * d.function_tolerance and o.gradient_tolerance == 10 * d.gradient_tolerance
    assert o.parameter_tolerance == 10 * d.parameter_tolerance


def test_runner_consumer_lines(tmp_path):
    """The statements VGGSfMRunner applies to the returned reconstruction (runner.py:552-560 add_point3D with an empty
    Track, :569-575 deregister_image, :996-1036 rename + camera rescale through images[id].camera_id /
    cameras[id].params / .width / .height, :596-609 calibration_matrix, :911 write) run on the stand-in."""
    c = cases()[0]
    rec = _build(c)
    n0 = rec.num_points3D()
    extra_xyz = np.array([[0.1, 0.2, 3.0], [0.3, -0.2, 4.0]])
    for k in range(2):
        rec.add_point3D(extra_xyz[k], rc.Track(), np.array([10, 20, 30 + k]))
    assert rec.num_points3D() == n0 + 2 and max(rec.point3D_ids()) == n0 + 2
    seen = sum(1 for p in rec.points3D.values() if any(e.image_id == 2 for e in p.track.elements))
    short = sum(1 for p in rec.points3D.values()
                if p.track.length() <= 2 and any(e.image_id == 2 for e in p.track.elements))
    rec.deregister_image(2)
    assert not rec.images[2].registered and rec.num_reg_images() == 4 and seen > 0
    assert rec.num_points3D() == n0 + 2 - short
    assert all(e.image_id != 2 for p in rec.points3D.values() for e in p.track.elements)
    names = [f"frame_{i:03d}.jpg" for i in range(5)]
    for pyimageid in rec.images:
        pyimage = rec.images[pyimageid]
        pycamera = rec.cameras[pyimage.camera_id]
        pyimage.name = names[pyimageid]
        params = pycamera.params.copy()
        params[0] *= 2.0
        params[1:3] = [960, 540]
        pycamera.params = params
        pycamera.width, pycamera.height = 1920, 1080
    Kc = rec.cameras[rec.images[0].camera_id].calibration_matrix()
    assert Kc[0, 0] == 2.0 * c["K"][0, 0, 0] and Kc[0, 2] == 960 and Kc[1, 2] == 540 and Kc[1, 1] == Kc[0, 0]
    rec.write(str(tmp_path))
    m = cio.read_model(str(tmp_path))
    assert sorted(m["images"]) == [0, 1, 3, 4] and m["images"][3]["name"] == "frame_003.jpg"
    assert m["cameras"][0]["width"] == 1920 and len(m["points3D"]) == rec.num_points3D()
    assert tuple(m["points3D"][n0 + 2]["rgb"]) == (10, 20, 31) and np.array_equal(m["points3D"][n0 + 1]["xyz"], extra_xyz[0])
    for pid, p in m["points3D"].items():          # surviving track elements still point at the right 2-D points
        for iid, idx in p["track"]:
            assert m["images"][iid]["point3D_ids"][idx] == pid


def test_normalize_matches_tensor_normalize():
    """Reconstruction.normalize (object graph) == bundle_adjustment.normalize (tensors): one Sim(3) rule, two holders."""
    from vggsfm_b200.bundle_adjustment import normalize
    c = cases()[1]
    rec = _build(c)
    rec.normalize(5.0, 0.1, 0.9, True)
    valid = np.nonzero(c["masks"].sum(0) >= 2)[0]
    E2, P2 = normalize(t(c["extr"]), t(c["pts"][valid]), 5.0, 0.1, 0.9)
    got_E = np.stack([rec.images[i].cam_from_world.matrix() for i in range(len(c["extr"]))])
    got_P = np.stack([rec.points3D[i + 1].xyz for i in range(len(valid))])
    assert np.abs(got_E - E2.numpy()).max() < 1e-12 and np.abs(got_P - P2.numpy()).max() < 1e-9 * np.abs(P2.numpy()).max()


def test_written_model_read_by_reference_reader(tmp_path):
    """cameras.bin / images.bin / points3D.bin written here are byte for byte the files the reference's reader
    (imc_helper.py:127-466) parsed into tests/golden/marshal_c_reader.npz (tools/make_golden_marshal.py), and what it
    parsed is the model."""
    g = np.load(os.path.join(GOLD, "marshal_c_reader.npz"))
    c = cases()[2]
    rec = _build(c)
    rec.set_point_colors(np.linspace(0, 1, rec.num_points3D())[:, None].repeat(3, 1))
    rec.write(str(tmp_path))
    for f in ("cameras", "images", "points3D"):
        with open(os.path.join(tmp_path, f + ".bin"), "rb") as fh:
            assert np.array_equal(np.frombuffer(fh.read(), dtype=np.uint8), g["bin_" + f]), f
    model = rec.to_model()
    assert list(g["cam_ids"]) == sorted(model["cameras"]) and list(g["img_ids"]) == sorted(model["images"])
    assert list(g["pt_ids"]) == sorted(model["points3D"])
    for k, cid in enumerate(g["cam_ids"]):
        assert g["cam_model"][k] == c["cam"] and tuple(g["cam_wh"][k]) == (1024, 768)
        assert np.array_equal(g["cam_params"][k], model["cameras"][cid]["params"])
    ends = np.cumsum(g["img_npts"])
    for k, iid in enumerate(g["img_ids"]):
        im = model["images"][iid]
        assert g["img_name"][k] == f"image_{iid}" and g["img_cam"][k] == im["camera_id"]
        assert np.allclose(g["img_R"][k], c["extr"][iid][:, :3], atol=1e-14) and np.array_equal(g["img_tvec"][k], c["extr"][iid][:, 3])
        lo, hi = ends[k] - g["img_npts"][k], ends[k]
        assert np.array_equal(g["img_xys"][lo:hi], im["xys"]) and np.array_equal(g["img_p3d"][lo:hi], im["point3D_ids"])
    ends = np.cumsum(g["pt_tracklen"])
    for k, pid in enumerate(g["pt_ids"]):
        p = model["points3D"][pid]
        assert np.array_equal(g["pt_xyz"][k], p["xyz"]) and np.array_equal(g["pt_rgb"][k], p["rgb"])
        lo, hi = ends[k] - g["pt_tracklen"][k], ends[k]
        assert [(int(a), int(b)) for a, b in g["pt_track"][lo:hi]] == p["track"]
