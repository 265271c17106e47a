"""Model-level parity of the three detector stacks on the same input (helper of
tests/test_reference_stack_gpu.py and tools/parity_report.py).

  A  the reference's unmodified Python stack on the reference's own CUDA extension (oracle/_ref)
  B  the reference's unmodified models/*.py on this package (install_as_reference_modules()), both
     with FAST_PATHS off (exact fp32 op sequence) and on (fused / bf16 eval kernels)
  C  spacap3d_b200.detector.VoteNetDetector

All with the reference's pretrained VoteNet weights (pretrained/PRETRAIN_VOTENET_*), TF32 off.

Element-wise criterion for the bf16 fast paths (north_star: "1e-2 for bf16 MLP"):
    |x - ref| <= TOL * |ref| + TOL * rms(ref)            for every element,
reported as  nerr = max |x - ref| / (|ref| + rms(ref))   (must be <= TOL = 1e-2).
"""
import contextlib

import numpy as np
import torch

SCENE_KW = {0: dict(use_height=False), 1: dict(use_height=True),
            7: dict(use_color=True, use_normal=True, use_height=True),
            132: dict(use_multiview=True, use_normal=True, use_height=True)}

INDEX_KEYS = ("sa1_inds", "sa2_inds", "fp2_inds", "seed_inds")
XYZ_KEYS = ("sa1_xyz", "sa2_xyz", "sa3_xyz", "sa4_xyz", "fp2_xyz", "seed_xyz")
FEATURE_KEYS = ("sa1_features", "sa2_features", "sa3_features", "sa4_features", "fp2_features", "seed_features",
                "vote_features")
PROPOSAL_KEYS = ("aggregated_vote_features", "objectness_scores", "center", "size_scores", "size_residuals",
                 "sem_cls_scores")


def make_batch(feature_dim, batch, n_points, seed0):
    from spacap3d_b200.scenes import make_scene
    kw = SCENE_KW[feature_dim]
    scenes = [make_scene(seed0 + i, n_points, with_replacement=(True if i == batch - 1 else None), **kw)
              for i in range(batch)]
    pc = torch.from_numpy(np.stack(scenes, 0))
    assert pc.shape[2] == 3 + feature_dim
    return pc


@contextlib.contextmanager
def exact_fp32(fast_paths):
    """TF32 off everywhere; FAST_PATHS of this package set as asked."""
    from spacap3d_b200 import pointnet2_modules as M
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, M.FAST_PATHS)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    M.FAST_PATHS = fast_paths
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, M.FAST_PATHS = old


@contextlib.contextmanager
def record_ball_query(utils_module, sink):
    """Record every ball-query index tensor `utils_module.ball_query` returns (reference:
    lib/pointnet2/pointnet2_utils.py:262-291 `ball_query = BallQuery.apply`)."""
    orig = utils_module.ball_query

    def wrapped(*a, **k):
        out = orig(*a, **k)
        sink.append(out.clone())
        return out
    utils_module.ball_query = wrapped
    try:
        yield
    finally:
        utils_module.ball_query = orig


def run_model(model, pc, utils_module):
    """forward -> (data_dict, [ball-query indices of SA1..SA4, vote aggregation])"""
    bq = []
    with torch.no_grad(), record_ball_query(utils_module, bq):
        out = model({"point_clouds": pc})
    return out, bq


def nerr(x, ref):
    """max over elements of |x-ref| / (|ref| + rms(ref))"""
    x, ref = x.double(), ref.double()
    rms = ref.pow(2).mean().sqrt().clamp_min(1e-30)
    return ((x - ref).abs() / (ref.abs() + rms)).max().item()


def max_rel_of_max(x, ref):
    return ((x.double() - ref.double()).abs().max() / ref.double().abs().max().clamp_min(1e-30)).item()


def compare(out, bq, ref, ref_bq, keys_float, report, tag, exact_indices=True):
    """Fill report[tag]: bit-equality of indices / coordinates / ball-query tables, nerr of floats."""
    r = report.setdefault(tag, {})
    for k in INDEX_KEYS + XYZ_KEYS:
        r[k + ":equal"] = bool(torch.equal(out[k], ref[k]))
    n_bq = min(len(bq), len(ref_bq)) if exact_indices else 4
    r["ball_query_tables_compared"] = n_bq
    for i in range(n_bq):
        r["ball_query[%d]:equal" % i] = bool(torch.equal(bq[i], ref_bq[i]))
    for k in keys_float:
        r[k + ":nerr"] = nerr(out[k], ref[k])
        r[k + ":bit_equal"] = bool(torch.equal(out[k], ref[k]))
    return r


def proposal_stage(proposal_module, vote_xyz, vote_features, utils_module):
    """Run only the proposal stage (vote aggregation SA + head + decode) on given votes."""
    bq = []
    with torch.no_grad(), record_ball_query(utils_module, bq):
        d = proposal_module(vote_xyz, vote_features, {})
    return d, bq


def reference_corners(stack, proposal_module, data_dict):
    """The reference's own decode (models/proposal_module.py:81-104 -> DC.param2obb_batch,
    data/scannet/model_util_scannet.py:165-173 -> utils/box_util.py:360-383 get_3d_box_batch) applied to
    `data_dict`'s center / size scores / residuals."""
    d = {k: data_dict[k] for k in ("center", "heading_scores", "heading_residuals", "size_scores", "size_residuals")}
    return stack.ProposalModule.decode_pred_box(proposal_module, d)


def collect(feature_dim, batch=8, n_points=40000, seed0=None, device="cuda:0"):
    """Run A, B (exact and fast) and C on one batch; return the comparison report (plain dict)."""
    from oracle import refstack
    import spacap3d_b200.pointnet2_utils as our_utils
    from spacap3d_b200.detector import VoteNetDetector
    seed0 = 7000 + 10 * feature_dim if seed0 is None else seed0
    pc = make_batch(feature_dim, batch, n_points, seed0).to(device)
    A = refstack.load_stack("reference")
    Bst = refstack.load_stack("dropin")
    mA = refstack.build_detector(A, feature_dim, device)
    mB = refstack.build_detector(Bst, feature_dim, device)
    mC = VoteNetDetector(input_feature_dim=feature_dim).to(device).eval()
    sd = torch.load(refstack.checkpoint_path(feature_dim), map_location="cpu")
    missing, unexpected = mC.load_state_dict(sd, strict=False)
    assert not missing and not unexpected, (missing, unexpected)

    report = {"feature_dim": feature_dim, "batch": batch, "n_points": n_points,
              "checkpoint": refstack.CHECKPOINTS[feature_dim]}
    floats = FEATURE_KEYS + ("vote_xyz",)
    with exact_fp32(False):
        oA, bqA = run_model(mA, pc, A.pointnet2_utils)
        oB, bqB = run_model(mB, pc, our_utils)
        compare(oB, bqB, oA, bqA, floats + PROPOSAL_KEYS, report, "B_exact_vs_A")
        report["B_exact_vs_A"]["aggregated_vote_inds:equal"] = bool(
            torch.equal(oB["aggregated_vote_inds"], oA["aggregated_vote_inds"]))
        report["B_exact_vs_A"]["bbox_corner:equal"] = bool(torch.equal(oB["bbox_corner"], oA["bbox_corner"]))
    with exact_fp32(True):
        for tag, model in (("B_fast_vs_A", mB), ("C_fast_vs_A", mC)):
            fast_vs_reference(report, tag, model, pc, oA, bqA, lambda d: reference_corners(A, mA.proposal, d))
    return report


def fast_vs_reference(report, tag, model, pc, oA, bqA, corners):
    """Fill report[tag]: `model` with the fast paths on, against the reference outputs oA / ball-query tables bqA
    of the same batch; `corners(data_dict)` is the reference's host box decode."""
    from spacap3d_b200 import pointnet2_utils as our_utils
    floats = FEATURE_KEYS + ("vote_xyz",)
    o, bq = run_model(model, pc, our_utils)
    r = compare(o, bq, oA, bqA, floats, report, tag, exact_indices=False)
    off, off_ref = o["vote_xyz"] - o["seed_xyz"], oA["vote_xyz"] - oA["seed_xyz"]
    r["vote_offset:nerr"] = nerr(off, off_ref)
    r["aggregated_vote_inds:equal_end_to_end"] = bool(
        torch.equal(o["aggregated_vote_inds"], oA["aggregated_vote_inds"]))
    r["aggregated_vote_inds:fraction_equal_end_to_end"] = float(
        (o["aggregated_vote_inds"] == oA["aggregated_vote_inds"]).float().mean())
    # every SA layer on the REFERENCE's inputs: the error of ONE fused 16-bit MLP (north_star's 1e-2 bound is
    # per MLP), without what earlier layers contributed
    xyz_in = pc[..., :3].contiguous()
    f_in = pc[..., 3:].transpose(1, 2).contiguous() if pc.shape[-1] > 3 else None
    with torch.no_grad():
        for i in (1, 2, 3, 4):
            _, f_out, _ = getattr(model.backbone_net, "sa%d" % i)(xyz_in, f_in)
            r["stage|sa%d_features:nerr" % i] = nerr(f_out, oA["sa%d_features" % i])
            xyz_in, f_in = oA["sa%d_xyz" % i], oA["sa%d_features" % i].clone()
    # proposal stage on the REFERENCE's votes (the vote FPS depends on feature values, so end to end
    # its picks may legitimately differ once vote_xyz differs in the last bits)
    d, bqp = proposal_stage(model.proposal, oA["vote_xyz"].clone(), oA["vote_features"].clone(), our_utils)
    r["proposal|aggregated_vote_inds:equal"] = bool(
        torch.equal(d["aggregated_vote_inds"], oA["aggregated_vote_inds"]))
    r["proposal|ball_query:equal"] = bool(torch.equal(bqp[0], bqA[4]))
    for k in PROPOSAL_KEYS:
        r["proposal|" + k + ":nerr"] = nerr(d[k], oA[k])
    r["proposal|bbox_mask:agree"] = float((d["bbox_mask"] == oA["bbox_mask"]).float().mean())
    r["proposal|sem_cls:agree"] = float((d["sem_cls"] == oA["sem_cls"]).float().mean())
    # N1: our on-device decode vs the reference's host decode on the SAME decoded parameters
    want = corners(d)
    r["proposal|bbox_corner_vs_get_3d_box_batch:equal"] = bool(torch.equal(d["bbox_corner"], want))
    r["proposal|bbox_corner_vs_get_3d_box_batch:maxabs"] = float((d["bbox_corner"] - want).abs().max())
    want_e2e = corners(o)
    r["bbox_corner_vs_get_3d_box_batch:equal"] = bool(torch.equal(o["bbox_corner"], want_e2e))


# ---- without the reference stack: the detector on the reference's point ops, pinned by digests ----------------------
# tests/golden/detector_ref.npz holds digests of every output of VoteNetDetector (seeded weights, the batches below, TF32
# off) run with the reference's op sequence and its nine point ops from `reference_ops()` -- the reference's own CUDA
# extension, or where it is not built the C oracle that tests/test_oracle_golden.py pins to that extension's stored
# outputs -- and the reference's host-side box decode as restated by bench.reference_host_decode
# (oracle/make_golden_detector.py).  None of this package's CUDA kernels computes them.  The reference's own Python
# modules and pretrained weights are not needed, so this is the reference's kernels under this package's module glue,
# not stack A: `collect_pinned` checks this package's exact mode against the digests bit for bit, then its fast mode
# against those exact outputs.
PINNED_KEYS = INDEX_KEYS + XYZ_KEYS + FEATURE_KEYS + ("vote_xyz",) + PROPOSAL_KEYS + (
    "aggregated_vote_inds", "bbox_corner", "bbox_mask", "sem_cls")


class OracleOnDevice:
    """bench.OracleOps for device tensors: arguments go to the host, results come back to `device`."""

    def __init__(self, device="cuda:0"):
        import bench
        self._ops, self._device = bench.OracleOps(), device

    def __getattr__(self, name):
        fn = getattr(self._ops, name)

        def call(*args):
            out = fn(*[a.detach().cpu() if torch.is_tensor(a) else a for a in args])
            return [o.to(self._device) for o in out] if isinstance(out, list) else out.to(self._device)
        return call


def reference_ops(device="cuda:0"):
    """-> (provider of the reference's nine point ops, what it is)."""
    try:
        from oracle.build_ref import load_ref
        return load_ref(), "reference CUDA extension (oracle/_ref)"
    except FileNotFoundError:
        return OracleOnDevice(device), "C oracle (pinned to the reference extension's outputs)"


def seeded_detector(feature_dim, batch=8, n_points=40000, seed0=None, device="cuda:0"):
    """-> (batch, VoteNetDetector with seeded weights in eval mode)."""
    from spacap3d_b200.detector import VoteNetDetector
    seed0 = 7000 + 10 * feature_dim if seed0 is None else seed0
    pc = make_batch(feature_dim, batch, n_points, seed0).to(device)
    torch.manual_seed(0)
    return pc, VoteNetDetector(input_feature_dim=feature_dim).to(device).eval()


def digests(out, bq):
    import cases
    d = {k: cases.sha(out[k].cpu().numpy()) for k in PINNED_KEYS}
    d.update({"ball_query[%d]" % i: cases.sha(t.cpu().numpy()) for i, t in enumerate(bq)})
    return d


def collect_pinned(feature_dim, golden, batch=8, n_points=40000, device="cuda:0"):
    """C (exact mode) against the pinned digests, then C (fast) against C (exact)."""
    import bench
    import spacap3d_b200.pointnet2_utils as our_utils
    pc, model = seeded_detector(feature_dim, batch, n_points, device=device)
    with exact_fp32(False):
        oE, bqE = run_model(model, pc, our_utils)
    report = {"feature_dim": feature_dim, "batch": batch, "n_points": n_points, "checkpoint": "seeded (torch seed 0)",
              "pinned_from": str(golden["meta/ops"])}
    r = report["C_exact_vs_pinned"] = {"ball_query_tables_compared": len(bqE)}
    for k, v in digests(oE, bqE).items():
        r[k + ":equal"] = v == str(golden["C%d/%s" % (feature_dim, k)])
    with exact_fp32(True):
        # box decode: the reference's host decode as restated by bench.reference_host_decode (not its own code)
        fast_vs_reference(report, "C_fast_vs_C_exact", model, pc, oE, bqE,
                          lambda d: bench.reference_host_decode(model.proposal, d))
    return report
