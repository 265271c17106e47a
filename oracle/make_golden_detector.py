"""Generate tests/golden/detector_ref.npz: digests of every output of spacap3d_b200.detector.VoteNetDetector (seeded
weights, the batches of tests/refparity.py, 1 / 7 / 132 input feature channels, TF32 off) run with the reference's
op sequence on the reference's nine point ops (refparity.reference_ops: its CUDA extension, or the C oracle pinned to
it) and the reference's host-side box decode (bench.reference_host_decode).  No CUDA kernel of this package runs.
Needs a GPU (the MLPs run on cuDNN, as they do in the package):

    python oracle/make_golden_detector.py OUT.npz        # then copy OUT.npz to tests/golden/detector_ref.npz

TEST INFRASTRUCTURE ONLY.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import bench  # noqa: E402
import refparity  # noqa: E402
import spacap3d_b200.pointnet2_utils as utils  # noqa: E402


def main(path):
    ops, what = refparity.reference_ops()
    out = {"meta/gpu": np.array(torch.cuda.get_device_name(0)), "meta/torch": np.array(torch.__version__),
           "meta/ops": np.array(what)}
    for c in (1, 7, 132):
        pc, model = refparity.seeded_detector(c)
        with refparity.exact_fp32(False), bench.swapped_ops(ops, host_decode=True):
            o, bq = refparity.run_model(model, pc, utils)
        out.update({"C%d/%s" % (c, k): np.array(v) for k, v in refparity.digests(o, bq).items()})
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes,", len(out), "arrays; point ops:", what)


if __name__ == "__main__":
    main(sys.argv[1])
