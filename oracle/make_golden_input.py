#!/usr/bin/env python
"""Golden vectors for the input-pipeline oracle (run in the build container, where /root/reference exists):
    python oracle/make_golden_input.py  ->  tests/golden/input_ref.npz

The point-data statements of `ScannetReferenceDataset.__getitem__` (lib/dataset.py:304-335, 361-431) are executed in
the reference's order around the REFERENCE'S OWN function bodies: random_sampling / rotx / roty / rotz
(utils/pc_utils.py), rotate_aligned_boxes_along_axis (data/scannet/model_util_scannet.py) and the dataset's
_translate method (lib/dataset.py:229-245) are cut out of the reference sources by AST and exec'd here -- their modules
cannot be imported (plyfile, trimesh, matplotlib, easydict, h5py are not installed).  np.random is seeded per case, so
the file also pins the RNG call order that spacap3d_b200.input_pipeline.draw_item restates."""
import ast
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402
import cases_input  # noqa: E402

REF = "/root/reference"


def _extract(path, names):
    tree = ast.parse(open(path).read())
    ns = {"np": np}
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name in names:
            mod = ast.Module(body=[node], type_ignores=[])
            exec(compile(mod, path, "exec"), ns)
    return [ns[n] for n in names]


random_sampling, rotx, roty, rotz = _extract(os.path.join(REF, "utils/pc_utils.py"),
                                             ["random_sampling", "rotx", "roty", "rotz"])
(rotate_aligned_boxes_along_axis,) = _extract(os.path.join(REF, "data/scannet/model_util_scannet.py"),
                                              ["rotate_aligned_boxes_along_axis"])
(_translate,) = _extract(os.path.join(REF, "lib/dataset.py"), ["_translate"])

MAX_NUM_OBJ = 128
MEAN_COLOR_RGB = np.array([109.8, 97.2, 83.8])
NYU40IDS = np.array([3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 23, 24, 25, 26, 27, 28, 29,
                     30, 31, 32, 33, 34, 35, 36, 37, 38, 39, 40])


def getitem(c):
    np.random.seed(c["seed"])
    mesh_vertices = c["verts"].copy()
    instance_labels, semantic_labels, instance_bboxes = c["inst"], c["sem"], c["bboxes"]
    if not c["use_color"]:
        point_cloud = mesh_vertices[:, 0:3]
    else:
        point_cloud = mesh_vertices[:, 0:6]
        point_cloud[:, 3:6] = (point_cloud[:, 3:6] - MEAN_COLOR_RGB) / 256.0
    if c["use_normal"]:
        normals = mesh_vertices[:, 6:9]
        point_cloud = np.concatenate([point_cloud, normals], 1)
    if c["use_multiview"]:
        point_cloud = np.concatenate([point_cloud, c["multiview"]], 1)
    floor_height = np.float32("nan")
    if c["use_height"]:
        floor_height = np.percentile(point_cloud[:, 2], 0.99)
        height = point_cloud[:, 2] - floor_height
        point_cloud = np.concatenate([point_cloud, np.expand_dims(height, 1)], 1)
    point_cloud, choices = random_sampling(point_cloud, c["P"], return_choices=True)
    instance_labels = instance_labels[choices]
    semantic_labels = semantic_labels[choices]

    target_bboxes = np.zeros((MAX_NUM_OBJ, 6))
    point_votes = np.zeros([c["P"], 3])
    point_votes_mask = np.zeros(c["P"])
    num_bbox = instance_bboxes.shape[0] if instance_bboxes.shape[0] < MAX_NUM_OBJ else MAX_NUM_OBJ
    target_bboxes[0:num_bbox, :] = instance_bboxes[:MAX_NUM_OBJ, 0:6]

    if c["augment"]:
        if np.random.random() > 0.5:
            point_cloud[:, 0] = -1 * point_cloud[:, 0]
            target_bboxes[:, 0] = -1 * target_bboxes[:, 0]
        if np.random.random() > 0.5:
            point_cloud[:, 1] = -1 * point_cloud[:, 1]
            target_bboxes[:, 1] = -1 * target_bboxes[:, 1]
        rot_angle = (np.random.random() * np.pi / 18) - np.pi / 36
        rot_mat = rotx(rot_angle)
        point_cloud[:, 0:3] = np.dot(point_cloud[:, 0:3], np.transpose(rot_mat))
        target_bboxes = rotate_aligned_boxes_along_axis(target_bboxes, rot_mat, "x")
        rot_angle = (np.random.random() * np.pi / 18) - np.pi / 36
        rot_mat = roty(rot_angle)
        point_cloud[:, 0:3] = np.dot(point_cloud[:, 0:3], np.transpose(rot_mat))
        target_bboxes = rotate_aligned_boxes_along_axis(target_bboxes, rot_mat, "y")
        rot_angle = (np.random.random() * np.pi / 18) - np.pi / 36
        rot_mat = rotz(rot_angle)
        point_cloud[:, 0:3] = np.dot(point_cloud[:, 0:3], np.transpose(rot_mat))
        target_bboxes = rotate_aligned_boxes_along_axis(target_bboxes, rot_mat, "z")
        point_cloud, target_bboxes = _translate(None, point_cloud, target_bboxes)

    for i_instance in np.unique(instance_labels):
        ind = np.where(instance_labels == i_instance)[0]
        if semantic_labels[ind[0]] in NYU40IDS:
            x = point_cloud[ind, :3]
            center = 0.5 * (x.min(0) + x.max(0))
            point_votes[ind, :] = center - x
            point_votes_mask[ind] = 1.0
    point_votes = np.tile(point_votes, (1, 3))
    assert point_cloud.dtype == np.float32, point_cloud.dtype
    return {"point_clouds": point_cloud.astype(np.float32), "choices": choices.astype(np.int64),
            "floor_height": np.float32(floor_height), "vote_label": point_votes.astype(np.float32),
            "vote_label_mask": point_votes_mask.astype(np.int64), "target_bboxes": target_bboxes,
            "center_label": target_bboxes.astype(np.float32)[:, 0:3], "num_bbox": np.array(num_bbox).astype(np.int64)}


def main():
    out = {}
    for name in cases_input.CASES:
        for k, v in getitem(cases_input.case(name)).items():
            # the point clouds (most of the file) are compared bit for bit: their digest is enough
            out["%s/%s" % (name, k)] = np.array(cases.sha(v)) if k == "point_clouds" else v
    # np.percentile on its own: many sizes / duplicate patterns
    for i, z in enumerate(cases_input.percentile_inputs()):
        out["percentile/%d" % i] = np.float32(np.percentile(z, 0.99))
    path = os.path.join(ROOT, "tests", "golden", "input_ref.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes,", len(out), "arrays; numpy", np.__version__)


if __name__ == "__main__":
    main()
