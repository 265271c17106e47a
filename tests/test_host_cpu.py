"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol that
include/spacap3d_ops.h declares, argument validation mirrors the reference (include/utils.h),
the module tree / state-dict keys match the reference checkpoints' (SURVEY F11), the product
never routes through the oracle, and the whole detector runs end to end on the CPU oracle
provider (this exercises every line of the module glue without a GPU)."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from spacap3d_b200 import _lib
    from spacap3d_b200.build import build_library
    build_library()
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "spacap3d_ops.h")).read()
    declared = set(re.findall(r"\b(spc_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 11
    for name in declared:
        assert hasattr(lib, name), name
    assert declared - {"spc_abi_version", "spc_last_error", "spc_fps_workspace_bytes", "spc_ball_query_workspace_bytes",
                       "spc_group_points_grad_workspace_bytes", "spc_bn_relu_workspace_bytes",
                       "spc_vote_labels_workspace_bytes"} == set(_lib.SIGNATURES)
    assert lib.spc_abi_version() == _lib.ABI_VERSION


def test_ctypes_signatures_match_the_header():
    """Every prototype of include/spacap3d_ops.h against the ctypes argument list the Python stub binds: same number
    of parameters, pointers where the header has pointers, int / float / size_t where it has scalars (a launch hint
    added on one side only would silently shift every later argument)."""
    import ctypes
    from spacap3d_b200 import _lib
    header = open(os.path.join(ROOT, "include", "spacap3d_ops.h")).read()
    header = re.sub(r"/\*.*?\*/", " ", header, flags=re.S)
    protos = dict(re.findall(r"\b(spc_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", header, flags=re.S))
    checked = 0
    for name, argtypes in _lib.SIGNATURES.items():
        params = [a.strip() for a in protos[name].replace("\n", " ").split(",")]
        assert len(params) == len(argtypes), (name, len(params), len(argtypes))
        for prm, ct in zip(params, argtypes):
            if "*" in prm:
                assert ct is ctypes.c_void_p, (name, prm, ct)
            elif prm.startswith("size_t"):
                assert ct is ctypes.c_size_t, (name, prm, ct)
            elif prm.startswith("float"):
                assert ct is ctypes.c_float, (name, prm, ct)
            elif prm.startswith(("int ", "unsigned")):
                assert ct in (ctypes.c_int, ctypes.c_uint), (name, prm, ct)
            elif prm.startswith(("uint64_t", "unsigned long long")):
                assert ct is ctypes.c_uint64, (name, prm, ct)
            elif prm.startswith("double"):
                assert ct is ctypes.c_double, (name, prm, ct)
            else:
                raise AssertionError("unhandled parameter %r of %s" % (prm, name))
            checked += 1
    assert checked > 300


def test_library_is_sm100a_and_uses_cluster_and_bulk_copy():
    out = subprocess.run(["cuobjdump", "-lelf", os.path.join(ROOT, "spacap3d_b200", "libspacap3d_ops.so")],
                         capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_argument_checks_mirror_reference():
    from spacap3d_b200 import _ext
    with pytest.raises(RuntimeError, match="CPU not supported"):
        _ext.furthest_point_sampling(torch.zeros(1, 4, 3), 2)
    with pytest.raises(RuntimeError, match="contiguous"):
        _ext.gather_points(torch.zeros(1, 4, 3).transpose(1, 2), torch.zeros(1, 2, dtype=torch.int32))
    with pytest.raises(RuntimeError, match="int"):
        _ext.group_points(torch.zeros(1, 3, 4), torch.zeros(1, 2, 2, dtype=torch.int64))
    with pytest.raises(RuntimeError, match="float"):
        _ext.three_nn(torch.zeros(1, 4, 3, dtype=torch.float64), torch.zeros(1, 4, 3))


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    from spacap3d_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.SpcError, match="no CPU"):
        _lib.load()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "spacap3d_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "liboracle" not in src, f


def test_state_dict_keys_match_reference_checkpoint_layout():
    from spacap3d_b200.detector import VoteNetDetector
    m = VoteNetDetector(input_feature_dim=1)
    keys = set(m.state_dict().keys())
    for k in ("backbone_net.sa1.mlp_module.layer0.conv.weight",
              "backbone_net.sa1.mlp_module.layer0.bn.bn.running_mean",
              "backbone_net.sa4.mlp_module.layer2.bn.bn.num_batches_tracked",
              "backbone_net.fp2.mlp.layer1.conv.weight", "vgen.conv3.bias", "vgen.bn2.running_var",
              "proposal.vote_aggregation.mlp_module.layer0.conv.weight", "proposal.proposal.6.bias"):
        assert k in keys, k
    assert len(keys) == 144                       # the reference's pretrained detectors hold 144 tensors
    assert m.state_dict()["backbone_net.sa1.mlp_module.layer0.conv.weight"].shape == (64, 4, 1, 1)
    assert sum(p.numel() for p in m.parameters()) == 953572
    ref_ckpt = "/root/reference/pretrained/PRETRAIN_VOTENET_XYZ/model.pth"
    if os.path.exists(ref_ckpt):                  # build container only
        r = m.load_state_dict(torch.load(ref_ckpt, map_location="cpu"), strict=False)
        assert not r.missing_keys and not r.unexpected_keys


def test_public_api_surface():
    from spacap3d_b200 import pointnet2_modules as M, pointnet2_utils as U, pytorch_utils as P
    for n in ("furthest_point_sample", "gather_operation", "three_nn", "three_interpolate",
              "grouping_operation", "ball_query", "QueryAndGroup", "GroupAll", "RandomDropout"):
        assert hasattr(U, n), n
    for n in ("PointnetSAModuleVotes", "PointnetFPModule", "PointnetSAModule", "PointnetSAModuleMSG",
              "PointnetSAModuleMSGVotes", "PointnetLFPModuleMSG"):
        assert hasattr(M, n), n
    for n in ("SharedMLP", "Conv1d", "Conv2d", "Conv3d", "FC", "BatchNorm1d", "BatchNorm2d",
              "BatchNorm3d", "BNMomentumScheduler", "set_bn_momentum_default"):
        assert hasattr(P, n), n
    mlp = [1, 64, 64, 128]
    M.PointnetSAModuleVotes(npoint=8, radius=0.2, nsample=4, mlp=mlp, use_xyz=True)
    assert mlp[0] == 4                            # the caller's list is mutated (+3), like the reference


def test_install_as_reference_modules():
    import spacap3d_b200
    spacap3d_b200.install_as_reference_modules()
    import pointnet2._ext as e                      # noqa: F401  the reference's import (pointnet2_utils.py:25-33)
    import pointnet2_utils                          # bare import after sys.path hack (pointnet2_modules.py:19-23)
    from lib.pointnet2.pointnet2_modules import PointnetSAModuleVotes, PointnetFPModule  # models/backbone_module.py:9
    assert pointnet2_utils.furthest_point_sample is not None and PointnetSAModuleVotes and PointnetFPModule


def test_detector_end_to_end_on_cpu_oracle_provider():
    """Runs the module glue (SA1-4, FP1-2, voting, proposal, decode) with the oracle as op provider;
    checks shapes, the reference's data_dict keys and the F10 prefix property."""
    sys.path.insert(0, ROOT)
    import bench
    from spacap3d_b200.detector import VoteNetDetector
    from spacap3d_b200.scenes import make_scene
    torch.manual_seed(0)
    model = VoteNetDetector(input_feature_dim=1).eval()
    pc = torch.from_numpy(np.stack([make_scene(5, 6000), make_scene(6, 6000, with_replacement=True)], 0))
    with bench.swapped_ops(bench.OracleOps(), host_decode=False), torch.no_grad():
        out = model({"point_clouds": pc})
        ref_boxes = bench.reference_host_decode(model.proposal, out)
    assert out["sa1_xyz"].shape == (2, 2048, 3) and out["fp2_features"].shape == (2, 256, 1024)
    assert out["bbox_corner"].shape == (2, 256, 8, 3) and out["bbox_corner"].dtype == torch.float64
    assert torch.equal(out["bbox_corner"], ref_boxes)      # device decode == reference host decode
    assert out["sem_cls_scores"].shape == (2, 256, 18) and out["size_residuals"].shape == (2, 256, 18, 3)
    assert torch.equal(out["sa2_inds"][0], torch.arange(1024, dtype=torch.int32))
    for k in ("seed_inds", "seed_xyz", "vote_xyz", "vote_features", "aggregated_vote_xyz",
              "aggregated_vote_inds", "objectness_scores", "center", "heading_scores",
              "heading_residuals", "size_scores", "bbox_mask", "bbox_sems", "sem_cls", "bbox_feature"):
        assert k in out, k


def test_bench_byte_and_flop_models_match_the_abi():
    """bench.py models algorithmic bytes / flops from the ctypes argument lists: every modelled entry point must
    exist in the ABI table and the model must not index past its arguments (an ABI change once silently dropped
    the fused-SA kernel from the roofline)."""
    import bench
    from spacap3d_b200 import _lib
    for table in (bench.ALGO_BYTES, bench.ALGO_FLOPS):
        for name, fn in table.items():
            assert name in _lib.SIGNATURES, name
            args = [1] * len(_lib.SIGNATURES[name])
            assert fn(args) >= 0
    for name in bench.ROOFLINE_BOUNDED:
        assert name in _lib.SIGNATURES, name
    # the fused-SA models of the two entry points agree on the same call
    a = [0, 0, 0, 0, 0, 0, 0, 1, 0.2, 0, 0, 0, 0, 8, 40000, 2048, 64, 64, 64, 128, 0, 0, 0]
    a_ex = a[:7] + [0, 0] + a[7:]
    assert bench.ALGO_BYTES["spc_sa_fused_forward"](a) == bench.ALGO_BYTES["spc_sa_fused_forward_ex"](a_ex)
    assert bench.ALGO_FLOPS["spc_sa_fused_forward"](a) == bench.ALGO_FLOPS["spc_sa_fused_forward_ex"](a_ex)


def test_bench_reference_arm_runs_without_a_gpu(tmp_path):
    """`bench.py --impl reference` must always print one JSON line: here (no GPU, hence no reference CUDA extension)
    it times the CPU oracle port on a bounded sample; the keys a reader of the line needs are all present, and
    --dump-outputs writes the detections of the last timed step."""
    import json
    import bench
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                         timeout=300, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "detector scenes/s @40k pts" and line["value"] > 0
    assert line["unit"] == "scenes/s" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["cores"] >= 0
    assert set(line["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"}
    assert "workload" in line["config"] and "model" not in line["config"]
    dumped = {p.name: np.load(p) for p in tmp_path.iterdir()}
    assert set(dumped) == {k + ".npy" for k in bench.RESULT_KEYS}
    assert dumped["bbox_corner.npy"].shape == (1, 256, 8, 3)
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in dumped.values())


def test_launch_options_are_thread_local_and_restored():
    """Launch hints travel per call from a thread-local context (the C ABI keeps no mutable state)."""
    import threading
    from spacap3d_b200 import _ext
    assert _ext._options.fps_algo == _ext.FPS_AUTO and _ext._options.sa_min_tiles == 0
    seen = {}

    def worker():
        seen["before"] = (_ext._options.fps_algo, _ext._options.sa_min_tiles)
        with _ext.launch_options(fps_algo=_ext.FPS_CLUSTER):
            seen["inside"] = _ext._options.fps_algo
    with _ext.launch_options(fps_algo=_ext.FPS_BUCKET, sa_min_tiles=16):
        t = threading.Thread(target=worker)
        t.start()
        t.join()
        assert (_ext._options.fps_algo, _ext._options.sa_min_tiles) == (_ext.FPS_BUCKET, 16)
        with _ext.launch_options(sa_min_tiles=4):
            assert _ext._options.sa_min_tiles == 4 and _ext._options.fps_algo == _ext.FPS_BUCKET
        assert _ext._options.sa_min_tiles == 16
        # a preference for the bucketed sampler only applies inside its size range
        assert _ext._fps_algo(40000) == _ext.FPS_BUCKET and _ext._fps_algo(2048) == _ext.FPS_AUTO
    assert seen == {"before": (_ext.FPS_AUTO, 0), "inside": _ext.FPS_CLUSTER}
    assert _ext._options.fps_algo == _ext.FPS_AUTO and _ext._options.sa_min_tiles == 0
    with pytest.raises(TypeError):
        _ext.launch_options(no_such_option=1)


def test_point_major_tag_follows_tensor_version():
    """attach_pm / get_pm_pair: the 16-bit copy is dropped when the fp32 tensor is edited in place or replaced."""
    import torch
    from spacap3d_b200.pointnet2_modules import attach_pm, get_pm, get_pm_pair
    t = torch.randn(2, 8, 5)
    pm = t.transpose(1, 2).contiguous().half()
    attach_pm(t, pm, pm.clone())
    hi, lo = get_pm_pair(t)
    assert hi is pm and lo is not None
    padded = torch.nn.functional.pad(pm, (0, 4))                 # channel dimension zero-padded to a multiple of 8
    assert get_pm(attach_pm(torch.randn(2, 8, 5), padded)) is padded
    t.mul_(2.0)
    assert get_pm(t) is None and get_pm_pair(t) == (None, None)
    assert get_pm(torch.randn(2, 8, 5)) is None
    u = torch.randn(2, 8, 5)
    attach_pm(u, torch.zeros(2, 6, 8).half())                    # wrong shape
    assert get_pm(u) is None


def test_folded_weight_caches_live_outside_the_module_dict():
    """ADVICE r1: nn.DataParallel's replicate() shallow-copies module __dict__s; the BN-folded weight caches must not
    ride along (replicas would share one cache object across devices and threads)."""
    import copy
    import torch
    from spacap3d_b200 import pointnet2_modules as M
    sa = M.PointnetSAModuleVotes(npoint=8, radius=0.3, nsample=16, mlp=[4, 64, 64, 128], use_xyz=True)
    c1 = M._cache_of(sa, M._FoldedMLP)
    assert M._cache_of(sa, M._FoldedMLP) is c1 and "_folded" not in sa.__dict__
    replica = copy.copy(sa)                                      # what replicate() does to the Python object
    assert M._cache_of(replica, M._FoldedMLP) is not c1
    M.invalidate_folded_caches(sa)
    assert M._cache_of(sa, M._FoldedMLP) is not c1


def test_reference_stack_imports_under_both_bindings():
    """oracle/refstack.py (test infrastructure): the reference's unmodified models import on top of this package
    ("dropin") and expose exactly the parameter tree of spacap3d_b200.detector; nothing leaks into sys.modules."""
    import sys
    from oracle import refstack
    if not refstack.available() and not os.path.isdir("/root/reference"):
        pytest.skip("baseline/_ref is not staged and /root/reference is absent")
    refstack._cache.pop("dropin", None)
    before = {k for k in sys.modules if k.split(".")[0] in refstack._TOP}
    B = refstack.load_stack("dropin")
    assert {k for k in sys.modules if k.split(".")[0] in refstack._TOP} == before     # nothing leaks
    assert "spacap3d_b200" in B.pointnet2_modules.__name__
    assert B.Pointnet2Backbone.__module__ == "models.backbone_module"       # the reference's own caller
    model = refstack.build_detector(B, 7, "cpu")                            # loads the pretrained checkpoint strictly
    from spacap3d_b200.detector import VoteNetDetector
    ours = VoteNetDetector(input_feature_dim=7)
    assert set(model.state_dict()) == set(ours.state_dict())
