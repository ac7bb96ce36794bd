"""Row f3 of SURVEY.md §8f: the textured .obj export (articulation3d_b200/export.py).  Structural tests (valid
triangulations, the file layout of utils/mesh_utils.py:_save, the geometry of the rotated copies) and, at the
end, byte-for-byte comparisons with the files the reference's own export writes (oracle/ref_export.py)."""
import os
import re

import numpy as np
import pytest

from articulation3d_b200 import OptConfig, export, synth

cv2 = pytest.importorskip("cv2")


def _poly_area(p):
    return 0.5 * abs(np.dot(p[:, 0], np.roll(p[:, 1], -1)) - np.dot(np.roll(p[:, 0], -1), p[:, 1]))


@pytest.mark.parametrize("shape", ["square", "L", "comb", "disc"])
def test_triangulation_covers_the_ring_exactly(shape):
    if shape == "square":
        ring = np.array([[0, 0], [4, 0], [4, 4], [0, 4]], float)
    elif shape == "L":
        ring = np.array([[0, 0], [6, 0], [6, 2], [2, 2], [2, 5], [0, 5]], float)
    elif shape == "comb":                                      # many reflex corners and collinear points
        ring = np.array([[0, 0], [1, 0], [2, 0], [9, 0], [9, 5], [8, 5], [8, 1], [6, 1], [6, 5], [5, 5], [5, 1], [3, 1],
                         [3, 5], [2, 5], [2, 1], [0, 1]], float)
    else:
        m = np.zeros((40, 50), np.uint8)
        cv2.circle(m, (25, 20), 13, 1, -1)
        ring = export.mask_to_polygons(m)[0]
    tri = export.triangulate(ring)
    assert tri.min() >= 0 and tri.max() < len(ring)
    areas = [_poly_area(ring[t]) for t in tri]
    assert min(areas) > 0
    assert sum(areas) == pytest.approx(_poly_area(ring), rel=1e-9)
    # same orientation for every triangle
    e1, e2 = ring[tri[:, 1]] - ring[tri[:, 0]], ring[tri[:, 2]] - ring[tri[:, 0]]
    cr = e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]
    assert all(c > 0 for c in cr) or all(c < 0 for c in cr)


def test_mask_to_polygons_returns_outer_rings_and_holes():
    m = np.zeros((30, 40), np.uint8)
    m[5:25, 5:35] = 1
    m[10:15, 10:20] = 0                                        # a hole: its ring is triangulated too, as in the reference
    rings = export.mask_to_polygons(m)
    assert len(rings) == 2
    assert export.mask_to_polygons(np.zeros((8, 8))) == []


def _parse_obj(path):
    meshes, cur = [], None
    for line in open(path):
        if line.startswith("# mesh"):
            cur = {"v": [], "vt": [], "f": [], "mtl": None}
            meshes.append(cur)
        elif line.startswith("v "):
            cur["v"].append(line.split()[1:])
        elif line.startswith("vt "):
            cur["vt"].append(line.split()[1:])
        elif line.startswith("usemtl"):
            cur["mtl"] = line.split()[1]
        elif line.startswith("f "):
            cur["f"].append([int(t.split("/")[0]) for t in line.split()[1:]])
    return meshes


def test_save_obj_model_layout_and_rotated_copies(tmp_path):
    cfg = OptConfig()
    preds, _ = synth.make_video(7, 2, 6, cfg, kinds=[0, 0])
    rng = np.random.RandomState(0)
    image = rng.randint(0, 255, size=(cfg.height, cfg.width, 3)).astype(np.uint8)
    path = export.save_obj_model(str(tmp_path), preds, 2, image=image, cfg=cfg)
    folder = os.path.dirname(path)
    assert os.path.basename(folder) == "frame_0002" and os.path.basename(path) == "arti_pred.obj"
    meshes = _parse_obj(path)
    assert len(meshes) == 1 + 5 + 2 + 1                        # object, 5 rotated copies, 2 axis markers, background
    text = open(path).read()
    assert text.startswith("mtllib arti_pred.mtl\n")
    assert re.search(r"^v -?\d+\.\d{10} -?\d+\.\d{10} -?\d+\.\d{10}$", text, re.M)          # ten decimals
    mtl = open(os.path.join(folder, "arti_pred.mtl")).read()
    base = 0
    for k, m in enumerate(meshes):
        assert m["mtl"] == f"arti_pred_uv_plane_{k}" and f"newmtl {m['mtl']}\n" in mtl
        png = cv2.imread(os.path.join(folder, "uv_maps", m["mtl"] + ".png"))
        assert png is not None and png.shape == (300, 300, 3)
        assert len(m["v"]) == len(m["vt"]) and len(m["f"]) % 2 == 0
        f = np.array(m["f"])
        assert f.min() >= base + 1 and f.max() <= base + len(m["v"])          # indices count over the whole file
        assert np.array_equal(f[0::2], f[1::2][:, ::-1])                      # double-sided
        base += len(m["v"])
    v = [np.array(m["v"], dtype=np.float64) for m in meshes]
    assert all(len(v[i]) == len(v[0]) for i in range(1, 6)) and len(v[6]) == len(v[7]) == 12
    # the copies are rigid rotations about the line through the two markers: distances to both ends are kept
    e0, e1 = v[6].mean(0), v[7].mean(0)
    for i in range(1, 6):
        for e in (e0, e1):
            np.testing.assert_allclose(np.linalg.norm(v[i] - e, axis=1), np.linalg.norm(v[0] - e, axis=1), rtol=0, atol=2e-5)
    # the grid arange(-1.8, 0.1, 0.45) ends at the identity: the last copy is the object itself
    np.testing.assert_allclose(v[5], v[0], atol=2e-6)
    assert np.abs(v[1] - v[0]).max() > 0.05
    # object and background share the plane: n.x = offset for both
    p = preds[2]
    b = int(np.asarray(p.scores).argmax())
    pl = p.pred_planes[b].numpy().astype(np.float64)
    pl = np.array([pl[0], -pl[2], pl[1]])
    for vv in (v[0], v[8]):
        np.testing.assert_allclose(vv @ (pl / np.linalg.norm(pl)), np.linalg.norm(pl), rtol=1e-5)


def test_frame_without_predictions_is_skipped(tmp_path, capsys):
    import torch
    from articulation3d_b200.structures import Boxes, Instances
    cfg = OptConfig()
    empty = Instances((cfg.height, cfg.width))
    empty.scores = np.zeros(0, dtype=np.float32)
    empty.pred_boxes = Boxes(torch.zeros(0, 4))
    empty.pred_masks = torch.zeros(0, cfg.height, cfg.width)
    empty.pred_planes = torch.zeros(0, 3)
    empty.pred_rot_axis = torch.zeros(0, 3)
    assert export.save_obj_model(str(tmp_path), [empty], 0, cfg=cfg) is None
    assert "no prediction" in capsys.readouterr().out


# ---------------------------------------------------------------------------------------------------
# pinned against the reference's own export (oracle/ref_export.py runs tools/inference.py:save_obj_model,
# utils/vis.py:get_single_image_mesh_arti and utils/mesh_utils.py:save_obj unmodified; only the outline and
# the triangulation routines, absent third-party code, are the product's)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["export_a", "export_b"])
def test_export_equals_reference_fixture(name, tmp_path, golden_dir):
    """Every file the export writes — .obj, .mtl, the nine 300x300 textures — byte for byte against the digest
    of what the reference's own export wrote for the same predictions and frame (tests/golden/export/*.json,
    generated by oracle/gen_golden.py --export)."""
    import json
    from oracle.gen_golden import export_case_inputs, export_digest
    with open(os.path.join(golden_dir, "export", f"{name}.json")) as f:
        want = json.load(f)
    preds, image, frame_id, axis_dir, webvis = export_case_inputs(name)
    obj = export.save_obj_model(str(tmp_path), preds, frame_id, image=image, axis_dir=axis_dir, webvis=webvis)
    got = export_digest(os.path.dirname(obj))
    assert got["_counts"] == want["_counts"] and got["_meshes"] == want["_meshes"]
    assert sorted(got) == sorted(want)
    for k in want:
        assert got[k] == want[k], f"{k} differs from the reference's file"
