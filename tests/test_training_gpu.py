"""Training mode (autograd through the unfused sm_100a kernels) against the reference's own CUDA
extension driving the same modules: forward values, input gradients and every parameter gradient.
Where that extension is not built (oracle/_ref), its nine entry points are served by the C oracle,
which tests/test_oracle_golden.py pins to the extension's stored outputs.
The reference's atomics make its gradients order-nondeterministic, hence rtol 1e-4 rather than
bitwise; both sides run cuDNN with TF32 disabled (SURVEY F8)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _stack(seed):
    from spacap3d_b200.pointnet2_modules import PointnetFPModule, PointnetSAModuleVotes
    torch.manual_seed(seed)
    sa1 = PointnetSAModuleVotes(npoint=256, radius=0.4, nsample=16, mlp=[4, 32, 32, 64], use_xyz=True, normalize_xyz=True)
    sa2 = PointnetSAModuleVotes(npoint=64, radius=0.8, nsample=16, mlp=[64, 64, 64, 128], use_xyz=True, normalize_xyz=True)
    fp = PointnetFPModule(mlp=[128 + 64, 64, 64])
    return torch.nn.ModuleList([sa1, sa2, fp]).to(DEV).train()


def _run(model, xyz, feats):
    sa1, sa2, fp = model
    x1, f1, i1 = sa1(xyz, feats)
    x2, f2, i2 = sa2(x1, f1)
    up = fp(x1, x2, f1, f2)
    loss = (up ** 2).mean() + (f2 ** 2).mean() + x2.sum() * 1e-3       # also sends a gradient into xyz via gather
    return loss, up, (i1, i2)


def test_train_step_matches_reference_extension(ref_ext):
    import bench
    import refparity
    provider = ref_ext if ref_ext is not None else refparity.OracleOnDevice(DEV)
    from spacap3d_b200.scenes import make_scene_xyz
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        xyz_np = np.stack([make_scene_xyz(90 + i, 3000) for i in range(3)], 0)
        g = torch.Generator(device="cpu").manual_seed(2)
        feats_np = torch.randn(3, 4, 3000, generator=g)
        outs = []
        for use_ref in (False, True):
            model = _stack(7)
            xyz = torch.from_numpy(xyz_np).to(DEV).requires_grad_(True)
            feats = feats_np.to(DEV).requires_grad_(True)
            if use_ref:
                with bench.swapped_ops(provider, host_decode=False):
                    loss, up, inds = _run(model, xyz, feats)
                    loss.backward()
            else:
                loss, up, inds = _run(model, xyz, feats)
                loss.backward()
            torch.cuda.synchronize()
            outs.append((loss.item(), up.detach(), inds, xyz.grad.clone(), feats.grad.clone(),
                         [p.grad.clone() for p in model.parameters()],
                         [b.clone() for n, b in model.named_buffers() if "running" in n]))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    ours, ref = outs
    assert torch.equal(ours[2][0], ref[2][0]) and torch.equal(ours[2][1], ref[2][1])   # FPS indices
    torch.testing.assert_close(ours[1], ref[1], rtol=1e-5, atol=1e-6)                  # forward features
    assert abs(ours[0] - ref[0]) <= 1e-5 * abs(ref[0])
    for a, b in [(ours[3], ref[3]), (ours[4], ref[4])] + list(zip(ours[5], ref[5])) + list(zip(ours[6], ref[6])):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-5 * max(1.0, b.abs().max().item()))


def test_reference_gradcheck_three_interpolate():
    """The reference's own test (lib/pointnet2/pointnet2_test.py:18-30), against our kernels."""
    from torch.autograd import gradcheck
    from spacap3d_b200 import pointnet2_utils
    feats = torch.randn(1, 2, 4, requires_grad=True).float().to(DEV)

    def interpolate_func(inputs):
        idx = torch.from_numpy(np.array([[[0, 1, 2], [1, 2, 3]]])).int().to(DEV)
        weight = torch.from_numpy(np.array([[[1, 1, 1], [2, 2, 2]]])).float().to(DEV)
        return pointnet2_utils.three_interpolate(inputs, idx, weight)

    assert gradcheck(interpolate_func, feats, atol=1e-1, rtol=1e-1)


def test_reference_smoke_block_msg_module():
    """The print-only smoke block of the reference (pointnet2_modules.py:505-525): forward + backward
    of a 2-scale MSG module; here with finite-ness and shape assertions."""
    from spacap3d_b200.pointnet2_modules import PointnetSAModuleMSG
    torch.manual_seed(1)
    xyz = torch.randn(2, 9, 3, device=DEV, requires_grad=True)
    xyz_feats = torch.randn(2, 6, 9, device=DEV, requires_grad=True)     # (B,C,N) as the module expects
    m = PointnetSAModuleMSG(npoint=2, radii=[5.0, 10.0], nsamples=[6, 3], mlps=[[6, 3], [6, 6]]).to(DEV)
    new_xyz, new_features = m(xyz, xyz_feats)
    assert new_xyz.shape == (2, 2, 3) and new_features.shape == (2, 9, 2)
    new_features.backward(torch.ones_like(new_features))
    assert torch.isfinite(new_features).all() and xyz_feats.grad is not None and torch.isfinite(xyz_feats.grad).all()
