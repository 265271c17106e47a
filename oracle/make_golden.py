"""Generate tests/golden/ref_ops.npz by running the REFERENCE's own CUDA extension
(oracle/_ref/pointnet2_ref_ext.so, built unmodified from /root/reference/lib/pointnet2/_ext_src
by oracle/build_ref.py) on the seeded cases in tests/cases.py.  Needs a GPU:

    gpurun -- python oracle/make_golden.py            # writes gpurun_out/golden/ref_ops.npz
    cp gpurun_out/golden/ref_ops.npz tests/golden/    # then commit

TEST INFRASTRUCTURE ONLY.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cases  # noqa: E402
from oracle.build_ref import load_ref  # noqa: E402


def compact(out):
    """Outputs the tests compare bit for bit are stored as their `cases.sha` digest (dtype, shape and bytes); the
    gradients, compared within a tolerance, are stored in full.  This keeps the file small."""
    return {k: v if k.endswith(("/grad", "/sha")) or k.startswith("meta/") else np.array(cases.sha(v))
            for k, v in out.items()}


def main():
    ref = load_ref()
    dev = torch.device("cuda:0")
    out = {}

    def cu(a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev)

    for name, (xyz, m) in cases.fps_cases().items():
        idx = ref.furthest_point_sampling(cu(xyz), int(m))
        out[f"fps/{name}/idx"] = idx.cpu().numpy()
        out[f"fps/{name}/sha"] = np.array(cases.sha(xyz, np.int64(m)))
    for name, (new_xyz, xyz, r, ns) in cases.ball_query_cases().items():
        idx = ref.ball_query(cu(new_xyz), cu(xyz), float(r), int(ns))
        out[f"ball_query/{name}/idx"] = idx.cpu().numpy()
        out[f"ball_query/{name}/sha"] = np.array(cases.sha(new_xyz, xyz, np.float32(r), np.int64(ns)))
    for name, (unknown, known) in cases.three_nn_cases().items():
        d2, idx = ref.three_nn(cu(unknown), cu(known))
        out[f"three_nn/{name}/dist2"] = d2.cpu().numpy()
        out[f"three_nn/{name}/idx"] = idx.cpu().numpy()
        out[f"three_nn/{name}/sha"] = np.array(cases.sha(unknown, known))
    for name, (pts, idx) in cases.gather_cases().items():
        o = ref.gather_points(cu(pts), cu(idx))
        g = cases.grad_for("gather/" + name, o.shape)
        gi = ref.gather_points_grad(cu(g), cu(idx), pts.shape[2])
        out[f"gather/{name}/out"] = o.cpu().numpy()
        out[f"gather/{name}/grad"] = gi.cpu().numpy()
        out[f"gather/{name}/sha"] = np.array(cases.sha(pts, idx, g))
    for name, (pts, idx) in cases.group_cases().items():
        o = ref.group_points(cu(pts), cu(idx))
        g = cases.grad_for("group/" + name, o.shape)
        gi = ref.group_points_grad(cu(g), cu(idx), pts.shape[2])
        out[f"group/{name}/out"] = o.cpu().numpy()
        out[f"group/{name}/grad"] = gi.cpu().numpy()
        out[f"group/{name}/sha"] = np.array(cases.sha(pts, idx, g))
    for name, (pts, idx, w) in cases.interp_cases().items():
        o = ref.three_interpolate(cu(pts), cu(idx), cu(w))
        g = cases.grad_for("interp/" + name, o.shape)
        gi = ref.three_interpolate_grad(cu(g), cu(idx), cu(w), pts.shape[2])
        out[f"interp/{name}/out"] = o.cpu().numpy()
        out[f"interp/{name}/grad"] = gi.cpu().numpy()
        out[f"interp/{name}/sha"] = np.array(cases.sha(pts, idx, w, g))
    torch.cuda.synchronize()
    out["meta/gpu"] = np.array(torch.cuda.get_device_name(0))
    out["meta/torch"] = np.array(torch.__version__)
    dst = os.path.join(ROOT, "gpurun_out", "golden")
    os.makedirs(dst, exist_ok=True)
    path = os.path.join(dst, "ref_ops.npz")
    np.savez_compressed(path, **compact(out))
    print("wrote", path, os.path.getsize(path), "bytes,", len(out), "arrays")


if __name__ == "__main__":
    main()
