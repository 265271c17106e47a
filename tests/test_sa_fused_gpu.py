"""Fused set-abstraction kernel (tcgen05) against
  (a) a torch emulation that applies the SAME fp16 roundings (tight: catches layout bugs), and
  (b) the reference op sequence in fp32 (FAST_PATHS off, TF32 off) at the tolerance north_star
      states for the fp16 MLP: rtol 1e-2 (measured against the tensor's max magnitude).
Shapes are the five SA layers of SpaCap3D (widths, nsample and radii exact, batch/points reduced)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
HALF = torch.float16          # spacap3d_b200._ext.HALF: storage type of the fused kernel's operands

# name: (n, Cf, npoint, radius, nsample, mlp)
LAYERS = {
    "sa1_xyz_height": (8192, 1, 512, 0.2, 64, [1, 64, 64, 128]),
    "sa1_xyz_only": (8192, 0, 512, 0.2, 64, [0, 64, 64, 128]),
    "sa1_rgb_normal_height": (8192, 7, 256, 0.2, 64, [7, 64, 64, 128]),
    "sa1_9ch_late_features": (4096, 9, 256, 0.2, 64, [9, 64, 64, 128]),       # in-line: 3 K steps, feature 8 read late
    "sa1_13ch_max_inline": (4096, 13, 256, 0.2, 32, [13, 64, 64, 128]),       # in-line: 4 K steps, the most it takes
    "sa1_14ch_projected": (4096, 14, 256, 0.2, 64, [14, 64, 64, 128]),        # one more channel: projected form
    "inline_wide": (4096, 4, 256, 0.3, 32, [4, 128, 128, 256]),               # in-line form at the wide widths (one CTA/SM, D2 ring)
    "inline_wide_ns16": (2048, 2, 128, 0.4, 16, [2, 128, 128, 128]),
    "sa1_ns16": (4096, 1, 256, 0.2, 16, [1, 64, 64, 128]),                    # 8 centres per tile: two 16-byte stores per lane
    "sa1_multiview": (4096, 132, 256, 0.3, 64, [132, 64, 64, 128]),
    "sa2": (2048, 128, 1024, 0.4, 32, [128, 128, 128, 256]),
    "sa3": (1024, 256, 512, 0.8, 16, [256, 128, 128, 256]),
    "sa4": (512, 256, 256, 1.2, 16, [256, 128, 128, 256]),
    "vote_agg": (1024, 256, 256, 0.3, 16, [256, 128, 128, 128]),
    # the remaining compiled (C1, C2, C3, nsample) kernels of each form, so that every one runs against the fp32 sequence
    "inline_wide_ns64": (4096, 4, 128, 0.3, 64, [4, 128, 128, 256]),
    "inline_wide_c256_ns16": (2048, 2, 256, 0.4, 16, [2, 128, 128, 256]),
    "inline_c128_ns64": (4096, 3, 128, 0.3, 64, [3, 128, 128, 128]),
    "inline_c128_ns32": (4096, 1, 256, 0.3, 32, [1, 128, 128, 128]),
    "projected_narrow_ns32": (4096, 16, 256, 0.3, 32, [16, 64, 64, 128]),
    "projected_narrow_ns16": (4096, 24, 256, 0.3, 16, [24, 64, 64, 128]),
    "projected_wide_ns64": (2048, 64, 256, 0.4, 64, [64, 128, 128, 256]),
    "projected_c128_ns64": (2048, 32, 256, 0.4, 64, [32, 128, 128, 128]),
    "projected_c128_ns32": (2048, 128, 512, 0.4, 32, [128, 128, 128, 128]),
}


def _module(mlp, npoint, radius, nsample, seed):
    from spacap3d_b200.pointnet2_modules import PointnetSAModuleVotes
    torch.manual_seed(seed)
    m = PointnetSAModuleVotes(npoint=npoint, radius=radius, nsample=nsample, mlp=list(mlp),
                              use_xyz=True, normalize_xyz=True).to(DEV)
    g = torch.Generator(device="cpu").manual_seed(seed + 1)
    for mod in m.modules():                      # non-trivial BN statistics / affine
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.running_mean.copy_(torch.randn(mod.num_features, generator=g) * 0.2)
            mod.running_var.copy_(torch.rand(mod.num_features, generator=g) + 0.5)
            mod.weight.data.copy_(torch.rand(mod.num_features, generator=g) + 0.5)
            mod.bias.data.copy_(torch.randn(mod.num_features, generator=g) * 0.1)
    return m.eval()


def _inputs(n, Cf, seed, B=2):
    from spacap3d_b200.scenes import make_scene_xyz
    xyz = torch.from_numpy(np.stack([make_scene_xyz(seed + i, n) for i in range(B)], 0)).to(DEV)
    g = torch.Generator(device="cpu").manual_seed(seed)
    feats = torch.randn(B, Cf, n, generator=g).to(DEV) if Cf > 0 else None
    return xyz, feats


@pytest.mark.parametrize("name", list(LAYERS.keys()))
def test_fused_matches_reference_sequence(name):
    from spacap3d_b200 import pointnet2_modules as M
    n, Cf, npoint, radius, nsample, mlp = LAYERS[name]
    m = _module(mlp, npoint, radius, nsample, seed=11)
    xyz, feats = _inputs(n, Cf, seed=31)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False      # SURVEY F8: fp32 reference must not run TF32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            M.FAST_PATHS = False
            ref_xyz, ref_feat, ref_inds = m(xyz, feats)
            M.FAST_PATHS = True
            new_xyz, new_feat, inds = m(xyz, feats)
    finally:
        M.FAST_PATHS = True
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    assert torch.equal(inds, ref_inds) and torch.equal(new_xyz, ref_xyz)      # indices bit-exact
    assert new_feat.shape == ref_feat.shape == (2, mlp[-1], npoint)
    # north_star: "1e-2 for bf16 MLP" -- checked ELEMENT-WISE: |err| <= 1e-2 |ref| + 1e-2 rms(ref) everywhere
    # (the kernel computes in fp16 with fp32 accumulation, ~8x tighter than bf16: measured 1-3e-3)
    rms = ref_feat.pow(2).mean().sqrt()
    nerr = ((new_feat - ref_feat).abs() / (ref_feat.abs() + rms)).max().item()
    assert nerr <= 1e-2, (name, nerr)
    scale = ref_feat.abs().max().item()
    assert (new_feat - ref_feat).abs().max().item() <= 2.5e-3 * scale, name
    assert (new_feat - ref_feat).abs().mean().item() <= 3e-4 * scale


@pytest.mark.parametrize("name", ["sa1_xyz_height", "sa2", "sa3", "vote_agg"])
def test_fused_matches_bf16_emulation(name):
    """Same roundings as the kernel (fp16 h1/h2/W1/W2, fp32 accumulate) => agreement to ~1e-3."""
    from spacap3d_b200 import _ext, pointnet2_modules as M, pointnet2_utils as U
    n, Cf, npoint, radius, nsample, mlp = LAYERS[name]
    m = _module(mlp, npoint, radius, nsample, seed=5)
    xyz, feats = _inputs(n, Cf, seed=77)
    with torch.no_grad():
        new_xyz, got, inds = m(xyz, feats)
        W0, b0, W1, b1, W2, b2 = M._FoldedMLP().get(m.mlp_module)
        idx = U.ball_query(radius, nsample, xyz, new_xyz)
        gx = U.grouping_operation(xyz.transpose(1, 2).contiguous(), idx)
        gx = (gx - new_xyz.transpose(1, 2).unsqueeze(-1)) / radius
        x = gx if feats is None else torch.cat([gx, U.grouping_operation(feats, idx)], 1)   # (B,K0,np,ns)
        if Cf > M.INLINE_MAX_FEATURES:
            # projected form: the per-point feature projection is a fp16 GEMM output (fp16 inputs,
            # fp32 accumulate, fp16 result); the xyz columns and the bias stay in fp32
            fb = feats.to(HALF).float()
            G = torch.einsum("ok,bkn->bon", W0[:, 3:].to(HALF).float(), fb).to(HALF).float()
            Gg = U.grouping_operation(G.contiguous(), idx)
            h1 = torch.relu(Gg + torch.einsum("ok,bkps->bops", W0[:, :3], gx) + b0[None, :, None, None])
        else:
            h1 = torch.relu(torch.einsum("ok,bkps->bops", W0, x) + b0[None, :, None, None])
        h1 = h1.to(HALF).float()
        h2 = torch.relu(torch.einsum("ok,bkps->bops", W1.float(), h1) + b1[None, :, None, None])
        h2 = h2.to(HALF).float()
        h3 = torch.einsum("ok,bkps->bops", W2.float(), h2)
        want = torch.relu(h3.max(-1).values + b2[None, :, None])
    scale = want.abs().max().item()
    assert (got - want).abs().max().item() <= 1e-3 * scale, name


def test_fused_not_used_in_training_or_with_grad():
    from spacap3d_b200 import pointnet2_modules as M
    n, Cf, npoint, radius, nsample, mlp = LAYERS["sa4"]
    m = _module(mlp, npoint, radius, nsample, seed=3)
    xyz, feats = _inputs(n, Cf, seed=9)
    feats.requires_grad_(True)
    _, f, _ = m(xyz, feats)                       # grad enabled -> reference sequence with autograd
    f.sum().backward()
    assert feats.grad is not None and torch.isfinite(feats.grad).all()
    m.train()
    with torch.no_grad():
        assert m._forward_fused(xyz, xyz[:, :npoint].contiguous(), feats) is None
