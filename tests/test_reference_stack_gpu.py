"""Model-level parity against the reference ITSELF, with its pretrained weights, at BASELINE size
(8 scenes x 40 000 points; C = 1 / 7 / 132 input feature channels = BASELINE configs 2 / 3 / 4).

  A  the reference's unmodified lib/pointnet2/*.py + models/*.py on the reference's own CUDA
     extension rebuilt for sm_100a (baseline/_ref + oracle/_ref; oracle/refstack.py)
  B  the SAME reference models/*.py (backbone_module.py:75-129, voting_module.py:34-61,
     proposal_module.py:57-158, SpaCapNet.py:47-74) after install_as_reference_modules(), i.e. the
     drop-in claim of north_star: callers unmodified, our modules and kernels underneath
  C  spacap3d_b200.detector.VoteNetDetector (the graph-friendly caller this repo ships)

Bars:
  * exact mode (FAST_PATHS off, TF32 off): B == A BIT FOR BIT -- every sampling index, coordinate,
    ball-query table, feature tensor, proposal score and decoded box corner.  (Stronger than the
    rtol 1e-5 north_star asks for fp32: the nine ops are bit-exact and the MLP is the same cuDNN call.)
  * fast mode (fused 16-bit tensor-core MLPs): all SA1-4 sampling indices, coordinates and ball-query
    tables still bit-equal (they do not depend on feature values); every feature tensor ELEMENT-WISE
        |x - ref| <= TOL |ref| + TOL rms(ref)
    with TOL = 1e-2 for each set-abstraction MLP (end to end AND on the reference's inputs) and for
    the proposal stage on the reference's votes; decoded corners equal utils/box_util.py
    get_3d_box_batch(DC.param2obb_batch(...)) bit for bit on the same decoded parameters.
  * the vote FPS depends on feature values (vote_xyz = seed_xyz + predicted offset), so once
    vote_xyz differs in the last bits its picks may differ: end to end only the fraction of equal
    picks is reported; on the reference's votes the picks are bit-equal.

Without the staged reference stack (its Python sources and checkpoints are not part of this repository), A is
replaced by tests/golden/detector_ref.npz: digests of every output of C with seeded weights run on the REFERENCE's
nine point ops (its CUDA extension, or the C oracle pinned to it) and a restatement of its host decode, computed
without any kernel of this package (oracle/make_golden_detector.py).  The exact mode of C must match them bit for
bit ("C_exact_vs_pinned"); the fast mode is then held to the bars above against those exact outputs
("C_fast_vs_C_exact", run for the C_fast_vs_A cases), with the box decode compared with bench.reference_host_decode,
this project's restatement of the reference's decode.  B, which needs the reference's models/*.py, skips.
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 1e-2
# The voting module (three more layers, then an L2 normalisation) amplifies the 3-5e-3 the four fused fp16 SA MLPs
# leave on its input: vote features / offsets are measured at 0.7-1.2e-2 end to end
# (profiles/r2_reference_stack_parity.txt); the FP / voting / proposal layers themselves are fp32-grade
# (tests/test_pm_linear_gpu.py) and add nothing measurable.
TOL_E2E_VOTES = 2e-2


def _stack_available():
    """True when the reference stack is staged; a staged stack whose extension does not load is an error, not a
    reason to fall back to the pinned outputs."""
    from oracle import refstack
    if not refstack.available():
        return False
    from oracle.build_ref import load_ref
    load_ref()
    return True


@pytest.fixture(scope="module", params=[1, 7, 132], ids=["xyz_C1", "rgb_normal_C7", "multiview_C132"])
def report(request):
    import numpy as np
    import refparity
    if _stack_available():
        return refparity.collect(request.param, batch=8, n_points=40000)
    golden = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "detector_ref.npz"))
    return refparity.collect_pinned(request.param, golden, batch=8, n_points=40000)


def _tag(report, tag):
    if tag in report:
        return report[tag]
    if tag == "C_fast_vs_A" and "C_fast_vs_C_exact" in report:       # no reference stack: see the module docstring
        return report["C_fast_vs_C_exact"]
    pytest.skip("%s needs the reference's models/*.py (baseline/_ref, not part of this repository)" % tag)


def test_exact_mode_equals_reference_bit_for_bit(report):
    r = report["B_exact_vs_A"] if "B_exact_vs_A" in report else report["C_exact_vs_pinned"]
    assert r["ball_query_tables_compared"] == 5
    bad = [k for k, v in r.items() if k.endswith("equal") and v is not True]
    assert not bad, bad


@pytest.mark.parametrize("tag", ["B_fast_vs_A", "C_fast_vs_A"])
def test_fast_mode_indices_bit_exact(report, tag):
    import refparity
    r = _tag(report, tag)
    for k in refparity.INDEX_KEYS + refparity.XYZ_KEYS:
        assert r[k + ":equal"] is True, k
    for i in range(4):
        assert r["ball_query[%d]:equal" % i] is True, i
    assert r["proposal|aggregated_vote_inds:equal"] is True
    assert r["proposal|ball_query:equal"] is True


@pytest.mark.parametrize("tag", ["B_fast_vs_A", "C_fast_vs_A"])
def test_fast_mode_features_elementwise(report, tag):
    r = _tag(report, tag)
    for i in (1, 2, 3, 4):
        assert r["sa%d_features:nerr" % i] <= TOL, (i, r["sa%d_features:nerr" % i])
        assert r["stage|sa%d_features:nerr" % i] <= TOL, (i, r["stage|sa%d_features:nerr" % i])
    for k in ("fp2_features", "seed_features"):
        assert r[k + ":nerr"] <= TOL, (k, r[k + ":nerr"])
    for k in ("vote_features", "vote_offset"):
        assert r[k + ":nerr"] <= TOL_E2E_VOTES, (k, r[k + ":nerr"])
    assert r["vote_xyz:nerr"] <= TOL
    import refparity
    for k in refparity.PROPOSAL_KEYS:
        assert r["proposal|" + k + ":nerr"] <= TOL, (k, r["proposal|" + k + ":nerr"])
    assert r["proposal|bbox_mask:agree"] >= 0.995 and r["proposal|sem_cls:agree"] >= 0.99


@pytest.mark.parametrize("tag", ["B_fast_vs_A", "C_fast_vs_A"])
def test_box_decode_equals_get_3d_box_batch(report, tag):
    """SURVEY row N1: the on-device decode against the reference's host decode (proposal_module.py:81-104)."""
    r = _tag(report, tag)
    assert r["proposal|bbox_corner_vs_get_3d_box_batch:equal"] is True, r["proposal|bbox_corner_vs_get_3d_box_batch:maxabs"]
    assert r["bbox_corner_vs_get_3d_box_batch:equal"] is True


def test_inplace_edit_between_layers_is_not_ignored():
    """ADVICE r1: the 16-bit point-major copy rides on the fp32 tensor as a tag; an in-place edit of the fp32 tensor
    must invalidate it (version counter) instead of being silently dropped by the next fast-path layer."""
    from spacap3d_b200.pointnet2_modules import PointnetSAModuleVotes, get_pm
    from spacap3d_b200.scenes import make_scene_xyz
    import numpy as np
    dev = "cuda:0"
    torch.manual_seed(0)
    sa1 = PointnetSAModuleVotes(npoint=512, radius=0.3, nsample=32, mlp=[0, 64, 64, 128], use_xyz=True,
                                normalize_xyz=True).to(dev).eval()
    sa2 = PointnetSAModuleVotes(npoint=256, radius=0.6, nsample=16, mlp=[128, 128, 128, 256], use_xyz=True,
                                normalize_xyz=True).to(dev).eval()
    xyz = torch.from_numpy(np.stack([make_scene_xyz(1, 4096), make_scene_xyz(2, 4096)], 0)).to(dev)
    with torch.no_grad():
        x1, f1, _ = sa1(xyz, None)
        assert get_pm(f1) is not None
        _, want_plain, _ = sa2(x1, f1)
        f1.mul_(0.0)                                   # in-place edit after the producer attached its copy
        assert get_pm(f1) is None
        _, got, _ = sa2(x1, f1)
        _, want, _ = sa2(x1, torch.zeros_like(f1))
    assert torch.equal(got, want)
    assert not torch.equal(got, want_plain)
