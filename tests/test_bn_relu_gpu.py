"""Training-mode BatchNorm + ReLU kernels (csrc/bn_relu.cu) against torch.nn.BatchNorm2d + ReLU in fp32
(the reference's pytorch_utils.Conv2d block, :11-36,39-64): forward values, running statistics,
num_batches_tracked, input / affine gradients; then a whole SA module, a channels_last block and a block with
B*C > 65535 trained with and without the fusion."""
import zlib

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

SHAPES = {
    "sa1_like": (3, 64, 512, 64),       # S = 32768, vectorised path, several position splits
    "sa3_like": (2, 256, 128, 16),
    "tiny_odd": (2, 5, 7, 3),           # S = 21: scalar path
    "one_channel": (4, 1, 33, 4),
    "big_mean": (2, 8, 64, 32),         # mean >> std: the shifted sums must not cancel
}


def _torch_ref(y, gamma, beta, rm, rv, momentum, eps, dz):
    y = y.clone().requires_grad_(True)
    gamma = gamma.clone().requires_grad_(True)
    beta = beta.clone().requires_grad_(True)
    z = torch.relu(torch.nn.functional.batch_norm(y, rm, rv, gamma, beta, True, momentum, eps))
    z.backward(dz)
    return z.detach(), y.grad, gamma.grad, beta.grad


@pytest.mark.parametrize("name", list(SHAPES.keys()))
def test_bn_relu_matches_torch(name):
    from spacap3d_b200 import _ext
    B, C, H, W = SHAPES[name]
    g = torch.Generator(device="cpu").manual_seed(zlib.crc32(name.encode()) % 1000)   # hash() is salted per process
    y = torch.randn(B, C, H, W, generator=g)
    if name == "big_mean":
        y = y * 0.01 + 50.0
    y = (y * (torch.rand(1, C, 1, 1, generator=g) + 0.5) + torch.randn(1, C, 1, 1, generator=g)).to(DEV)
    gamma = (torch.rand(C, generator=g) + 0.5).to(DEV)
    beta = (torch.randn(C, generator=g) * 0.3).to(DEV)
    rm0, rv0 = torch.randn(C, generator=g).to(DEV), (torch.rand(C, generator=g) + 0.5).to(DEV)
    dz = torch.randn(B, C, H, W, generator=g).to(DEV)
    momentum, eps = 0.1, 1e-5
    old = torch.backends.cudnn.enabled
    torch.backends.cudnn.enabled = False          # ATen's own fp32 batch-norm kernels as the reference
    try:
        rm_ref, rv_ref = rm0.clone(), rv0.clone()
        z_ref, dy_ref, dg_ref, db_ref = _torch_ref(y, gamma, beta, rm_ref, rv_ref, momentum, eps, dz)
    finally:
        torch.backends.cudnn.enabled = old
    rm, rv = rm0.clone(), rv0.clone()
    z, mean, invstd = _ext.bn_relu_train_forward(y, gamma, beta, rm, rv, momentum, eps)
    dy, dg, db = _ext.bn_relu_train_backward(dz, y, gamma, beta, mean, invstd)
    # big_mean: |mean|/std = 5000, so one ulp of the fp32 batch mean (4e-6) is already 4e-4 standard deviations --
    # two correct fp32 implementations differ by that much; everywhere else 1e-5
    tol = 1e-3 if name == "big_mean" else 1e-5
    torch.testing.assert_close(z, z_ref, rtol=tol, atol=tol)
    torch.testing.assert_close(rm, rm_ref, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(rv, rv_ref, rtol=1e-3 if name == "big_mean" else 1e-5, atol=1e-7)
    # The ReLU mask is recomputed from y: an element whose normalised value is within rounding of 0 may land on
    # the other side than in ATen (its gradient then differs by the full dz*gamma*invstd).  Compare dy away from
    # the kink, and require the kink set to be tiny; the channel sums absorb the few flipped elements.
    zlin = torch.nn.functional.batch_norm(y, None, None, gamma, beta, True, 0.0, eps)
    stable = zlin.abs() > 50 * tol
    assert (~stable).float().mean().item() < 200 * tol        # ~N(0,1) density around 0
    scale = max(1.0, dy_ref.abs().max().item())
    torch.testing.assert_close(torch.where(stable, dy, dy_ref), dy_ref, rtol=10 * tol, atol=10 * tol * scale)
    # channel sums: equal up to fp32 summation error plus whatever the elements at the kink can contribute
    xhat = torch.nn.functional.batch_norm(y, None, None, None, None, True, 0.0, eps)
    slack_g = ((dz * xhat).abs() * ~stable).sum(dim=(0, 2, 3))
    slack_b = (dz.abs() * ~stable).sum(dim=(0, 2, 3))
    assert ((dg - dg_ref).abs() <= slack_g + 1e-4 * max(1.0, dg_ref.abs().max().item())).all()
    assert ((db - db_ref).abs() <= slack_b + 1e-4 * max(1.0, db_ref.abs().max().item())).all()


def test_sa_module_training_step_same_with_and_without_fusion():
    """One optimiser-free training step of an SA module: loss, every gradient, running statistics and
    num_batches_tracked agree between the fused BN+ReLU path and the plain module sequence."""
    from spacap3d_b200 import pytorch_utils
    from spacap3d_b200.pointnet2_modules import PointnetSAModuleVotes
    from spacap3d_b200.scenes import make_scene_xyz
    xyz = torch.from_numpy(np.stack([make_scene_xyz(60 + i, 4000) for i in range(3)], 0)).to(DEV)
    feats = torch.randn(3, 4, 4000, generator=torch.Generator().manual_seed(1)).to(DEV)
    old_tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    res = []
    try:
        for fused in (True, False):
            pytorch_utils.FUSED_BN_RELU_TRAINING = fused
            torch.manual_seed(3)
            m = PointnetSAModuleVotes(npoint=256, radius=0.4, nsample=16, mlp=[4, 32, 32, 64], use_xyz=True,
                                      normalize_xyz=True).to(DEV).train()
            f = feats.clone().requires_grad_(True)
            _, out, _ = m(xyz, f)
            loss = (out ** 2).mean()
            loss.backward()
            res.append((loss.item(), out.detach(), f.grad, [p.grad for p in m.parameters()],
                        {n: b.clone() for n, b in m.named_buffers()}))
    finally:
        pytorch_utils.FUSED_BN_RELU_TRAINING = True
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old_tf32
    (l1, o1, g1, p1, b1), (l2, o2, g2, p2, b2) = res
    assert abs(l1 - l2) <= 1e-5 * abs(l2)
    torch.testing.assert_close(o1, o2, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(g1, g2, rtol=1e-3, atol=1e-5 * max(1.0, g2.abs().max().item()))
    for a, b in zip(p1, p2):
        torch.testing.assert_close(a, b, rtol=1e-3, atol=1e-5 * max(1.0, b.abs().max().item()))
    assert b1.keys() == b2.keys()
    for k in b1:
        if b1[k].dtype.is_floating_point:
            torch.testing.assert_close(b1[k], b2[k], rtol=1e-5, atol=1e-6)
        else:
            assert torch.equal(b1[k], b2[k]), k


@pytest.mark.parametrize("ns", [16, 32, 64])
def test_bn_relu_maxpool_matches_torch(ns):
    """BatchNorm + ReLU + max over nsample in one kernel pair vs batch_norm -> relu -> max_pool2d, with
    ball-query style duplicated slots (ties) and all-negative groups."""
    from spacap3d_b200 import _ext
    B, C, npnt = 3, 24, 200
    g = torch.Generator(device="cpu").manual_seed(ns)
    y = torch.randn(B, C, npnt, ns, generator=g)
    y[:, :, :, ns // 2:] = y[:, :, :, :1]                  # padding: second half repeats slot 0 (exact ties)
    y[:, :, ::7] -= 6.0                                     # some groups entirely below zero after BN
    y = (y * (torch.rand(1, C, 1, 1, generator=g) + 0.5)).contiguous().to(DEV)
    gamma = (torch.rand(C, generator=g) + 0.5).to(DEV)
    gamma[::5] *= -1.0                                      # negative scale: the max is the smallest input
    beta = (torch.randn(C, generator=g) * 0.3).to(DEV)
    rm0, rv0 = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    dpool = torch.randn(B, C, npnt, generator=g).to(DEV)
    old = torch.backends.cudnn.enabled
    torch.backends.cudnn.enabled = False
    try:
        yr, gr, br = y.clone().requires_grad_(True), gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
        rm_ref, rv_ref = rm0.clone(), rv0.clone()
        z = torch.relu(torch.nn.functional.batch_norm(yr, rm_ref, rv_ref, gr, br, True, 0.1, 1e-5))
        pooled_ref = torch.nn.functional.max_pool2d(z, kernel_size=[1, ns]).squeeze(-1)
        pooled_ref.backward(dpool)
    finally:
        torch.backends.cudnn.enabled = old
    rm, rv = rm0.clone(), rv0.clone()
    pooled, argmax, ymax, mean, invstd = _ext.bn_relu_maxpool_train_forward(y, gamma, beta, rm, rv, 0.1, 1e-5)
    dy, dg, db = _ext.bn_relu_maxpool_train_backward(dpool, argmax, ymax, y, gamma, beta, mean, invstd)
    torch.testing.assert_close(pooled, pooled_ref.detach(), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(rm, rm_ref, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(rv, rv_ref, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(dy, yr.grad, rtol=1e-4, atol=1e-4 * max(1.0, yr.grad.abs().max().item()))
    torch.testing.assert_close(dg, gr.grad, rtol=1e-4, atol=1e-4 * max(1.0, gr.grad.abs().max().item()))
    torch.testing.assert_close(db, br.grad, rtol=1e-4, atol=1e-4 * max(1.0, br.grad.abs().max().item()))


@pytest.mark.parametrize("case", ["channels_last", "BC72000-pool"])
def test_conv_block_fuses_any_layout_and_batch(case, monkeypatch):
    """A conv block whose output is not contiguous (a channels_last model) or has B*C > 65535 rows (the kernels then
    run in slices of at most 65535 / C batch rows) takes the fused kernels too, with the same results as the plain
    module sequence.  beta = 10 keeps every normalised value far from the ReLU kink, where the two may round apart."""
    from spacap3d_b200 import _lib, pytorch_utils
    pool = case.endswith("-pool")
    B, Cin, C, H, W = (3, 4, 24000, 2, 16) if pool else (2, 8, 16, 64, 32)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, Cin, H, W, generator=g).to(DEV)
    wout = torch.randn((B, C, H) if pool else (B, C, H, W), generator=g).to(DEV)
    names, real = [], _lib.call

    def spy(name, *args):
        names.append(name)
        return real(name, *args)

    monkeypatch.setattr(_lib, "call", spy)
    # fp32 convolutions: with TF32 the conv backward rounds dy to 10 mantissa bits, which turns the fp32 rounding
    # difference between the two BatchNorm implementations into 1e-3-level differences of the input gradient
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    res = []
    try:
        for fused in (True, False):
            pytorch_utils.FUSED_BN_RELU_TRAINING = fused
            torch.manual_seed(7)
            m = pytorch_utils.Conv2d(Cin, C, bn=True).to(DEV).train()
            torch.nn.init.constant_(m.bn.bn.bias, 10.0)
            xi = x.clone()
            if not pool:
                m = m.to(memory_format=torch.channels_last)
                xi = xi.to(memory_format=torch.channels_last)
                assert not m.conv(xi).is_contiguous()
            xi.requires_grad_(True)
            out = m(xi, max_pool_last_dim=pool)
            (out * wout).sum().backward()
            res.append((out.detach(), xi.grad, [p.grad for p in m.parameters()],
                        {n: b.clone() for n, b in m.named_buffers()}))
    finally:
        pytorch_utils.FUSED_BN_RELU_TRAINING = True
    fwd = "spc_bn_relu_maxpool_train_forward" if pool else "spc_bn_relu_train_forward"
    assert names.count(fwd) == 1 and not [n for n in names if "_sync" in n], names
    (o1, g1, p1, b1), (o2, g2, p2, b2) = res
    torch.testing.assert_close(o1, o2, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(g1, g2, rtol=1e-3, atol=1e-5 * max(1.0, g2.abs().max().item()))
    for a, b in zip(p1, p2):
        torch.testing.assert_close(a, b, rtol=1e-3, atol=1e-5 * max(1.0, b.abs().max().item()))
    for k in b1:
        torch.testing.assert_close(b1[k], b2[k], rtol=1e-5, atol=1e-6)
