"""Training under torch.autocast("cuda", dtype=torch.bfloat16): the bf16 twins of the grouping, interpolation and fused
BatchNorm + ReLU (+ max-pool) kernels, and the modules that route to them.

  * Exact kernel tests: the dyadic data of test_exact_training_kernels.py and test_sync_bn.py is bf16-representable
    (BatchNorm inputs mu + 2^e t need at most 8 significant bits, gradients are k/8, weights k/16), and on it the fp32
    value of every output is exact.  A bf16 output is rounded once from that value, so it must equal the float64
    reference rounded to bf16, by torch.equal; fp32 outputs (statistics, dgamma / dbeta, gradients of grouping and
    interpolation before _ext's cast) must equal the reference itself.  The exceptions of those files carry over:
    running_var within one fp32 ulp, dy within its bound plus one bf16 ulp when M is not a power of two.
  * The max-pool compares bf16-ROUNDED values: a case where slots differ only below bf16 resolution checks that the
    lowest one wins, as F.max_pool2d on the bf16 tensor.
  * Random data against torch's own bf16 sequence (cuDNN BatchNorm on the bf16 conv output, ReLU, max_pool2d).
  * The detector's training step under autocast: eager against a replayed CUDA graph, the bf16 entry points reached,
    the fp32 step unchanged, and loss and gradients against the fp32 step under the bars REL_BAR_LOSS / REL_BAR_GRAD.
CPU-only tests check the preconditions, the bf16 launch plans the cases reach and the dtype checks of _ext.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_exact_training_kernels import (BN_CASES, BN_MOMENTUM, DEV, FP32_UNITS, GROUP_CASES, INTERP_CASES, POOL_CASES,
                                         _bn_dev, _bn_reference, _cdiv, _check_bn_outputs, _constants, _expect_equal,
                                         _gen, _k8, _poison, grad_route, make_bn, make_group_idx, make_interp_idx_w)
from test_sync_bn import SYNC_CASES, SYNC_POOL_CASES, K as SYNC_K, _local_sums, _slices, make_sync_bn

BF16 = torch.bfloat16


def _bf16_exact(t):
    return torch.equal(t.to(BF16).double(), t.double())


def _to_bf16(t):
    """An fp32-exact value rounded once to bf16 (the float64 -> float step is exact)."""
    return t.float().to(BF16)


# ---- bf16 launch plans (group.cu; the staged budgets count bytes, bf16 rows take half) ------------------------------
def plan_group_bf16(K, B, C, N, S):
    """plan_group of the bf16 forward: (staged, CT, nchunks)."""
    row = 2 * N
    staged = row <= K["GP_ROW_BUDGET"] and N > 0
    CT = max(1, min(K["GP_CT_BYTES"] // row, C, K["GP_CT_MAX"])) if staged else 4
    ctiles = _cdiv(C, CT)
    nchunks = 1
    while B * ctiles * nchunks < K["GP_WAVES"] * K["kNumSMs"] and S // (nchunks * 2) >= K["GP_CHUNK_MIN"]:
        nchunks *= 2
    chunk = (_cdiv(S, nchunks) + 3) & ~3
    return staged, CT, _cdiv(S, chunk)


def plan_group_grad_bf16(K, C, N, S):
    """plan_group_grad with bf16 grad_out rows staged: (H, Sp, CT, lists_smem)."""
    H = _cdiv(S, K["GG_PART_MAX"])
    Sp = _cdiv(_cdiv(S, H), 8) * 8
    H = _cdiv(S, Sp)
    Np = (N + 1 + 3) // 4 * 4
    CT = max(1, min(K["GG_CT_BYTES"] // (Sp * 2), K["GG_CT_MAX"], C))
    return H, Sp, CT, CT * Sp * 2 + Sp * 2 + Np * 4 <= K["GG_LISTS_SMEM"]


# (id, B, C, N, npoint, nsample, hubs), as GROUP_CASES
BF16_GROUP_CASES = [c for c in GROUP_CASES if c[0] in (
    "csr-ct4-h1", "csr-ct2-nobulk", "csr-h2-nobulk", "csr-h2-global", "csr-h3-ragged-smem", "ex-fallback-n3000-c5",
    "gather-n8193-1tile", "gather-ragged-tile", "gather-16tiles", "unstaged-vec4", "unstaged-scalar", "c5-80k-sa1-feat",
    "c5-80k-sa2", "c5-200k-sa1-feat", "c5-200k-sa2")] + [
    ("bf16-csr-ct3", 2, 7, 1000, 320, 30, 8),           # S=9600: bf16 rows of Sp=9600 -> CT=3
    ("bf16-staged-nobulk-n1001", 2, 3, 1001, 128, 16, 4),   # 2002-byte rows: staged without the bulk copy
    ("bf16-staged-n102400", 1, 2, 102400, 256, 16, 8),  # exactly the 200 KB budget: staged (fp32: unstaged)
    ("bf16-unstaged-n102401", 1, 2, 102401, 256, 16, 8),  # one point more: unstaged
]


def bf16_group_branches(K, case):
    name, B, C, N, npoint, ns, hubs = case
    S = npoint * ns
    br = set()
    staged, CT, _ = plan_group_bf16(K, B, C, N, S)
    if staged:
        bulk = all(((b * C + c0) * N * 2) % 16 == 0 and (min(CT, C - c0) * N * 2) % 16 == 0
                   for b in range(B) for c0 in range(0, C, CT))
        br.add("fwd staged" + ("" if bulk else ", no bulk copy"))
        if 4 * N > K["GP_ROW_BUDGET"]:
            br.add("fwd staged only in bf16")
    else:
        br.add("fwd unstaged")
    br.add("fwd vec4" if S % 4 == 0 else "fwd scalar")
    r = grad_route(K, C, N, C >= K["EX_MIN_C"])
    if r.startswith("atomic"):
        br.add("atomic" + (" C<4" if C < K["EX_MIN_C"] else ""))
    elif r == "gather":
        br.add("gather")
    else:
        H, Sp, GCT, smem = plan_group_grad_bf16(K, C, N, S)
        br |= {"csr CT=%d" % GCT, "csr H=%d" % min(H, 3), "csr lists " + ("smem" if smem else "global")}
    return br


BF16_GROUP_BRANCHES = {"fwd staged", "fwd staged, no bulk copy", "fwd staged only in bf16", "fwd unstaged", "fwd vec4",
                       "fwd scalar", "atomic C<4", "atomic", "gather", "csr CT=1", "csr CT=2", "csr CT=3", "csr CT=4",
                       "csr H=1", "csr H=2", "csr H=3", "csr lists smem", "csr lists global"}


# ---- CPU-only --------------------------------------------------------------------------------------------------------
def test_bf16_cases_reach_every_plan_branch():
    """With the plan constants read from the sources, the bf16 grouping cases reach the staged / unstaged threshold of
    bf16 rows (102 400 points against 51 200 for fp32) on both sides, the staging without a bulk copy, the list-based
    backward with 1, 2 and >= 3 partitions and every channel tile CT, the point-owned gather and the atomic kernel."""
    K = _constants()
    assert K["GP_ROW_BUDGET"] // 2 == 102400
    reached = set()
    for c in BF16_GROUP_CASES:
        reached |= bf16_group_branches(K, c)
    assert BF16_GROUP_BRANCHES <= reached, sorted(BF16_GROUP_BRANCHES - reached)


def test_bf16_cases_meet_preconditions():
    """Every input of the exact bf16 cases is bf16-representable, and the sums stay exact in fp32."""
    for c in BF16_GROUP_CASES:
        assert c[4] * c[5] * 8 < FP32_UNITS
    for c in INTERP_CASES:
        _, w = make_interp_idx_w(c)
        assert _bf16_exact(torch.from_numpy(w)) and 3 * c[4] * 2 ** 7 < FP32_UNITS
    k8 = torch.arange(-8, 9, dtype=torch.float64) / 8
    assert _bf16_exact(k8)
    for cases, pool in ((BN_CASES, False), (POOL_CASES, True)):
        for c in cases:
            if _bn_dev(c) != "cpu":
                # generator parameters: mu = k/16 with |k| <= 64, a = 2^e with e in [-3, 2], |t| <= 2, so y is a
                # multiple of 2^-4 below 4 + 8 = 12 in magnitude: 192 units < 2^8; dz is k/2 or k, |k| <= 2
                assert (4 + 2 ** 2 * 2) * 16 < 2 ** 8
                continue
            d = make_bn(c, "cpu", pool=pool)
            assert _bf16_exact(d["y"]) and _bf16_exact(d["dz"]), c["id"]
    for cases, pool in ((BF16_SYNC_CASES, False), (BF16_SYNC_POOL_CASES, True)):
        for c in cases:
            d, _, _ = make_sync_bn(c, pool)
            assert d["y"].device.type == "cpu" and _bf16_exact(d["y"]) and _bf16_exact(d["dz"]), c["id"]


@pytest.mark.parametrize("dtype", [torch.float16, torch.float64])
def test_ext_rejects_other_dtypes(dtype):
    """fp32 and bf16 are the storage types; anything else raises the fp32 check's message, as before."""
    from spacap3d_b200 import _ext
    i3 = torch.zeros(1, 2, 2, dtype=torch.int32)
    w = torch.zeros(1, 2, 3)
    x = torch.zeros(1, 3, 4, dtype=dtype)
    for fn, args, name in ((_ext.group_points, (x, i3), "points"),
                           (_ext.group_points_grad, (torch.zeros(1, 3, 2, 2, dtype=dtype), i3, 4), "grad_out"),
                           (_ext.three_interpolate, (x, torch.zeros(1, 2, 3, dtype=torch.int32), w), "points"),
                           (_ext.three_interpolate_grad, (torch.zeros(1, 3, 2, dtype=dtype),
                                                          torch.zeros(1, 2, 3, dtype=torch.int32), w, 4), "grad_out"),
                           (_ext.bn_relu_train_forward, (x, torch.ones(3), torch.zeros(3), None, None, 0.1, 1e-5), "y"),
                           (_ext.bn_relu_maxpool_train_forward, (torch.zeros(1, 3, 2, 16, dtype=dtype), torch.ones(3),
                                                                 torch.zeros(3), None, None, 0.1, 1e-5), "y")):
        with pytest.raises(RuntimeError, match="%s must be a float tensor" % name):
            fn(*args)
    with pytest.raises(RuntimeError, match="float"):
        _ext.gather_points(torch.zeros(1, 3, 4, dtype=BF16), torch.zeros(1, 2, dtype=torch.int32))


def test_fused_path_decides_on_the_conv_output_dtype():
    """A model cast wholesale to bf16 keeps torch's BatchNorm (its parameters are not fp32); fp32 BatchNorm
    parameters pass the module-level checks, whatever the block input's dtype."""
    from spacap3d_b200 import pytorch_utils as pt
    blk = pt.Conv2d(4, 8, bn=True).train()
    assert blk._fusable
    bn = blk.bn[0]
    assert bn.weight.dtype == torch.float32
    blk_bf = pt.Conv2d(4, 8, bn=True).train().bfloat16()
    assert blk_bf.bn[0].weight.dtype == BF16
    cuda_like = type("T", (), {"is_cuda": True})()        # the check reads only is_cuda of the block input
    assert blk._fused_training_ok(cuda_like) and not blk_bf._fused_training_ok(cuda_like)


# ---- exact kernel tests (GPU) ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", BF16_GROUP_CASES, ids=[c[0] for c in BF16_GROUP_CASES])
def test_group_points_bf16_exact(case):
    """bf16 group_points == the gather; the fp32 gradient of both bf16 backward entry points == the float64
    scatter_add_, and _ext's bf16 gradient == that rounded once."""
    from spacap3d_b200 import _ext, _lib
    name, B, C, N, npoint, ns, hubs = case
    S = npoint * ns
    idx = torch.from_numpy(make_group_idx(case)).to(DEV)
    g = _gen(name, DEV)
    points = _k8((B, C, N), g, DEV).to(BF16)
    li = idx.view(B, 1, S).long().expand(B, C, S)
    _poison((B, C, S))
    out = _ext.group_points(points, idx)
    assert out.dtype == BF16
    _expect_equal(out.view(B, C, S), torch.gather(points, 2, li), "group_points")
    del out
    go = _k8((B, C, npoint, ns), g, DEV).to(BF16)
    want = torch.zeros(B, C, N, dtype=torch.float64, device=DEV).scatter_add_(2, li, go.view(B, C, S).double())
    _poison((B, C, N))
    got = _ext.group_points_grad(go, idx, N)
    assert got.dtype == BF16
    _expect_equal(got, _to_bf16(want), "_ext.group_points_grad")
    stream = torch.cuda.current_stream().cuda_stream
    got = torch.full((B, C, N), float("nan"), device=DEV)
    _lib.call("spc_group_points_grad_bf16", go.data_ptr(), idx.data_ptr(), B, C, N, npoint, ns, got.data_ptr(), stream)
    _expect_equal(got, want, "spc_group_points_grad_bf16")
    nbytes = _lib.load().spc_group_points_grad_workspace_bytes(B, N, npoint, ns)
    ws = torch.empty((nbytes + 3) // 4, dtype=torch.int32, device=DEV)
    got.fill_(float("nan"))
    _lib.call("spc_group_points_grad_ex_bf16", go.data_ptr(), idx.data_ptr(), B, C, N, npoint, ns, got.data_ptr(),
              ws.data_ptr(), nbytes, stream)
    _expect_equal(got, want, "spc_group_points_grad_ex_bf16")


@pytest.mark.gpu
@pytest.mark.parametrize("case", INTERP_CASES, ids=[c[0] for c in INTERP_CASES])
def test_three_interpolate_bf16_exact(case):
    from spacap3d_b200 import _ext, _lib
    name, B, C, m, n = case
    idx_np, w_np = make_interp_idx_w(case)
    idx, w = torch.from_numpy(idx_np).to(DEV), torch.from_numpy(w_np).to(DEV)
    g = _gen(name, DEV)
    points, go = _k8((B, C, m), g, DEV).to(BF16), _k8((B, C, n), g, DEV).to(BF16)
    li = idx.view(B, 1, 3 * n).long().expand(B, C, 3 * n)
    if n:
        want = (torch.gather(points.double(), 2, li).view(B, C, n, 3) * w.double()[:, None]).sum(-1)
        _poison((B, C, n))
        out = _ext.three_interpolate(points, idx, w)
        assert out.dtype == BF16
        _expect_equal(out, _to_bf16(want), "three_interpolate")
    want = torch.zeros(B, C, m, dtype=torch.float64, device=DEV).scatter_add_(
        2, li, (go.double()[..., None] * w.double()[:, None]).reshape(B, C, 3 * n))
    _poison((B, C, m))
    got = _ext.three_interpolate_grad(go, idx, w, m)
    assert got.dtype == BF16
    _expect_equal(got, _to_bf16(want), "three_interpolate_grad")
    got32 = torch.full((B, C, m), float("nan"), device=DEV)
    _lib.call("spc_three_interpolate_grad_bf16", go.data_ptr(), idx.data_ptr(), w.data_ptr(), B, C, n, m,
              got32.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _expect_equal(got32, want, "spc_three_interpolate_grad_bf16")


def _check_bf16_outputs(ref, got, what):
    """bf16 outputs against the reference rounded once to bf16 (dy: within its bound plus one bf16 ulp when M is not a
    power of two); fp32 outputs as _check_bn_outputs."""
    f32 = {}
    for k, v in got.items():
        if v.dtype != BF16:
            f32[k] = v
            continue
        want = ref[k].to(DEV)
        if k == "dy" and not ref["exact_dy"]:
            bound = ref["dy_err"].to(DEV)
            ulp = 2.0 ** (torch.floor(torch.log2(want.abs() + bound)) - 7)
            err = (v.double() - want).abs()
            assert bool((err <= bound + ulp).all()), (what, "dy", float((err - bound - ulp).max()))
        else:
            _expect_equal(v, _to_bf16(want), "%s %s" % (what, k))
    _check_bn_outputs(ref, f32, what)


def _dev_bf16(d, offset=False):
    y = _to_bf16(d["y"].to(DEV))
    if offset:                                        # 2 bytes past 8-byte alignment: the scalar kernels
        store = torch.empty(y.numel() + 1, dtype=BF16, device=DEV)
        store[1:] = y.flatten()
        y = store[1:].view(y.shape)
        assert y.data_ptr() % 8 == 2
    f = lambda k: d[k].float().to(DEV)                              # noqa: E731
    return y, f("gamma"), f("beta"), f("rm"), f("rv"), _to_bf16(d["dz"].to(DEV))


@pytest.mark.gpu
@pytest.mark.parametrize("c", BN_CASES, ids=[c["id"] for c in BN_CASES])
def test_bn_relu_train_bf16_exact(c):
    from spacap3d_b200 import _ext
    d = make_bn(c, _bn_dev(c))
    ref = _bn_reference(d)
    y, gamma, beta, rm, rv, dz = _dev_bf16(d, c.get("offset", False))
    _poison(y.shape)
    z, mean, invstd = _ext.bn_relu_train_forward(y, gamma, beta, rm, rv, BN_MOMENTUM, d["eps"])
    dy, dgamma, dbeta = _ext.bn_relu_train_backward(dz, y, gamma, beta, mean, invstd)
    assert z.dtype == dy.dtype == BF16 and mean.dtype == dgamma.dtype == torch.float32
    _check_bf16_outputs(ref, dict(z=z, mean=mean, invstd=invstd, rm=rm, rv=rv, dy=dy, dgamma=dgamma, dbeta=dbeta),
                        c["id"])


@pytest.mark.gpu
@pytest.mark.parametrize("c", POOL_CASES, ids=[c["id"] for c in POOL_CASES])
def test_bn_relu_maxpool_bf16_exact(c):
    from spacap3d_b200 import _ext
    d = make_bn(c, _bn_dev(c), pool=True)
    ref = _bn_reference(d, pool=True)
    y, gamma, beta, rm, rv, dpool = _dev_bf16(d)
    pooled, argmax, ymax, mean, invstd = _ext.bn_relu_maxpool_train_forward(y, gamma, beta, rm, rv, BN_MOMENTUM,
                                                                            d["eps"])
    _poison(y.shape)
    dy, dgamma, dbeta = _ext.bn_relu_maxpool_train_backward(dpool, argmax, ymax, y, gamma, beta, mean, invstd)
    _check_bf16_outputs(ref, dict(pooled=pooled, argmax=argmax, ymax=ymax, mean=mean, invstd=invstd, rm=rm, rv=rv,
                                  dy=dy, dgamma=dgamma, dbeta=dbeta), c["id"])


BF16_SYNC_CASES = [c for c in SYNC_CASES if c["id"] in (
    "2r-vec-pow2", "3r-vec-pow2", "2r-uneven-3+2", "3r-scalar-S6", "2r-1+3-means", "2r-empty-rank")]
BF16_SYNC_POOL_CASES = [c for c in SYNC_POOL_CASES if c["id"] in (
    "2r-ns16-pow2", "2r-ns32-uneven-3+2", "3r-ns64-uneven", "3r-ns16-empty-rank")]


def _run_sync_bf16(c, pool):
    """test_sync_bn's emulated ranks on bf16 y / dz: every rank fills its row of a zeroed buffer, their sum is the
    all-reduce, and every rank's outputs are checked against the float64 evaluation over the whole batch."""
    from spacap3d_b200 import _ext
    d, _, _ = make_sync_bn(c, pool)
    ref = _bn_reference(d, pool=pool)
    C, ranks = c["C"], c["ranks"]
    R = len(ranks)
    sls = _slices(ranks)
    f = lambda k: d[k].float().to(DEV)                              # noqa: E731
    y, dz, gamma, beta = _to_bf16(d["y"].to(DEV)), _to_bf16(d["dz"].to(DEV)), f("gamma"), f("beta")
    bufs = []
    for r, sl in enumerate(sls):
        buf = torch.zeros(R, C, SYNC_K, dtype=torch.float64, device=DEV)
        _ext.bn_relu_sync_stats(y[sl].contiguous(), buf[r])
        bufs.append(buf)
    rows = sum(bufs)
    outs, saved = [], []
    for r, sl in enumerate(sls):
        yr = y[sl].contiguous()
        rm, rv = f("rm"), f("rv")
        if pool:
            pooled, argmax, ymax, mean, invstd = _ext.bn_relu_maxpool_sync_forward(yr, gamma, beta, rm, rv, BN_MOMENTUM,
                                                                                  d["eps"], rows)
            fwd = dict(pooled=pooled, argmax=argmax, ymax=ymax)
        else:
            z, mean, invstd = _ext.bn_relu_sync_forward(yr, gamma, beta, rm, rv, BN_MOMENTUM, d["eps"], rows)
            fwd = dict(z=z)
        fwd.update(mean=mean, invstd=invstd, rm=rm, rv=rv)
        outs.append(fwd)
        saved.append((yr, mean, invstd))
    bufs, local = [], []
    for r, sl in enumerate(sls):
        yr, mean, invstd = saved[r]
        buf = torch.zeros(R, C, SYNC_K, dtype=torch.float64, device=DEV)
        dzr = dz[sl].contiguous()
        if pool:
            local.append(_ext.bn_relu_maxpool_sync_backward_reduce(dzr, outs[r]["ymax"], yr, gamma, beta, mean, invstd,
                                                                   buf[r]))
        else:
            local.append(_ext.bn_relu_sync_backward_reduce(dzr, yr, gamma, beta, mean, invstd, buf[r]))
        bufs.append(buf)
    rows = sum(bufs)
    for r, sl in enumerate(sls):
        yr, mean, invstd = saved[r]
        dzr = dz[sl].contiguous()
        if pool:
            dy = _ext.bn_relu_maxpool_sync_backward(dzr, outs[r]["argmax"], outs[r]["ymax"], yr, gamma, beta, mean,
                                                    invstd, rows)
        else:
            dy = _ext.bn_relu_sync_backward(dzr, yr, gamma, beta, mean, invstd, rows)
        dbeta_r, dgamma_r = _local_sums(d, ref, sl, pool)
        rref = dict(ref, dbeta=dbeta_r, dgamma=dgamma_r)
        for k in ("z", "pooled", "argmax", "ymax", "dy", "dy_err"):
            if k in ref:
                rref[k] = ref[k][sl]
        got = dict(outs[r], dgamma=local[r][0], dbeta=local[r][1])
        if ranks[r]:
            got["dy"] = dy
        _check_bf16_outputs(rref, got, "%s rank %d" % (c["id"], r))


@pytest.mark.gpu
@pytest.mark.parametrize("c", BF16_SYNC_CASES, ids=[c["id"] for c in BF16_SYNC_CASES])
def test_bn_relu_sync_bf16_exact(c):
    _run_sync_bf16(c, pool=False)


@pytest.mark.gpu
@pytest.mark.parametrize("c", BF16_SYNC_POOL_CASES, ids=[c["id"] for c in BF16_SYNC_POOL_CASES])
def test_bn_relu_maxpool_sync_bf16_exact(c):
    _run_sync_bf16(c, pool=True)


@pytest.mark.gpu
def test_maxpool_ties_below_bf16_resolution_keep_the_lowest_slot():
    """gamma = 1 and beta = 100: the kernel's z = fma(xhat, 1, 100) is reproduced exactly by fp32 torch ops, and near
    100 the bf16 spacing (0.5) merges slots whose fp32 values differ.  pooled and the winning slot must be those of
    F.max_pool2d on the bf16-rounded tensor, which keeps the first of equal values."""
    from spacap3d_b200 import _ext
    torch.manual_seed(1)
    B, C, npoint, ns = 2, 3, 96, 16
    y = (torch.randn(B, C, npoint, ns, device=DEV) * 0.2).to(BF16)
    gamma, beta = torch.ones(C, device=DEV), torch.full((C,), 100.0, device=DEV)
    pooled, argmax, ymax, mean, invstd = _ext.bn_relu_maxpool_train_forward(y, gamma, beta, None, None, 0.1, 1e-5)
    zf = (y.float() - mean.view(1, C, 1, 1)) * invstd.view(1, C, 1, 1) + 100.0
    zb = torch.relu(zf.to(BF16))
    want, ind = F.max_pool2d(zb.view(B * C, npoint, ns), kernel_size=(1, ns), return_indices=True)
    assert bool((zf.argmax(-1) != zb.float().argmax(-1)).any()), "no group with a tie below bf16 resolution"
    assert torch.equal(pooled.view(B * C, npoint), want.view(B * C, npoint))
    assert torch.equal(argmax.view(B * C, npoint).long(), ind.view(B * C, npoint) % ns)
    assert torch.equal(ymax, y.gather(-1, argmax.long().unsqueeze(-1)).squeeze(-1))


# ---- random data against torch's own bf16 sequence ----------------------------------------------------------------------
def _bf16_ulp(t):
    return 2.0 ** (torch.floor(torch.log2(t.float().abs().clamp_min(2.0 ** -126))) - 7)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(4, 128, 1024, 32), (4, 64, 2048, 64), (4, 256, 1024, 1)],
                         ids=["sa2-ns32", "sa1-ns64", "fp-1x1"])
def test_bn_relu_matches_torch_bf16_sequence(shape):
    """cuDNN BatchNorm on a bf16 y (fp32 math, one rounding) + ReLU (+ max_pool2d on the bf16 tensor): z and pooled
    within one bf16 ulp, the winning slot equal wherever torch's rounded maximum leads the runner-up by more than two
    ulps (a one-ulp rounding difference of either side cannot reorder those), running statistics close."""
    from spacap3d_b200 import _ext
    torch.manual_seed(sum(shape))
    B, C = shape[:2]
    y = (torch.randn(shape, device=DEV) * 2 + torch.randn(1, C, 1, 1, device=DEV)).to(BF16)
    gamma, beta = torch.rand(C, device=DEV) + 0.5, torch.randn(C, device=DEV) * 0.5
    rm_t, rv_t = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    zt = torch.relu(F.batch_norm(y, rm_t, rv_t, gamma, beta, training=True, momentum=0.1, eps=1e-5))
    assert zt.dtype == BF16
    rm, rv = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    if shape[-1] > 1:
        pooled, argmax, _, _, _ = _ext.bn_relu_maxpool_train_forward(y, gamma, beta, rm, rv, 0.1, 1e-5)
        pt = F.max_pool2d(zt, kernel_size=(1, shape[-1])).squeeze(-1)
        assert bool(((pooled.float() - pt.float()).abs() <= _bf16_ulp(pt)).all())
        top2 = zt.float().topk(2, dim=-1).values
        clear = (top2[..., 0] - top2[..., 1]) > 2 * _bf16_ulp(top2[..., 0])
        assert bool(clear.float().mean() > 0.5)
        assert torch.equal(argmax.long()[clear], zt.float().argmax(-1)[clear])
    else:
        z, mean, invstd = _ext.bn_relu_train_forward(y, gamma, beta, rm, rv, 0.1, 1e-5)
        # one bf16 ulp, plus the fp32 cancellation of gamma * xhat + beta near the ReLU's 0, where the two fp32
        # evaluations may fall on either side of 0 (a few fp32 ulps of the terms)
        xh = (y.float() - mean.view(1, C, 1, 1)) * invstd.view(1, C, 1, 1)
        terms = (xh * gamma.view(1, C, 1, 1)).abs() + beta.view(1, C, 1, 1).abs()
        bound = torch.maximum(_bf16_ulp(zt), _bf16_ulp(z)) + 2.0 ** -20 * terms
        assert bool(((z.float() - zt.float()).abs() <= bound).all())
    torch.testing.assert_close(rm, rm_t, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(rv, rv_t, rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
def test_grouping_and_interpolation_match_torch_index_ops():
    """bf16 grouping equals torch.gather; bf16 interpolation equals the fp32 kernel on the same values rounded once
    (same arithmetic, one rounding), and is within one bf16 ulp of the float64 evaluation; the bf16 backward passes
    agree with the fp32 ones on the same bf16 gradients up to fp32 summation order and the final rounding."""
    from spacap3d_b200 import _ext
    torch.manual_seed(3)
    B, C, N, npoint, ns = 4, 128, 4096, 2048, 32
    points = torch.randn(B, C, N, device=DEV).to(BF16)
    idx = torch.randint(0, N, (B, npoint, ns), device=DEV, dtype=torch.int32)
    out = _ext.group_points(points, idx)
    li = idx.view(B, 1, -1).long().expand(B, C, -1)
    assert torch.equal(out.view(B, C, -1), torch.gather(points, 2, li))
    go = torch.randn(B, C, npoint, ns, device=DEV).to(BF16)
    g16, g32 = _ext.group_points_grad(go, idx, N), _ext.group_points_grad(go.float(), idx, N)
    assert g16.dtype == BF16
    assert bool(((g16.float() - g32).abs() <= _bf16_ulp(g32) + 1e-5 * g32.abs().max()).all())
    m, n = 2048, 4096
    feats = torch.randn(B, 256, m, device=DEV).to(BF16)
    iidx = torch.randint(0, m, (B, n, 3), device=DEV, dtype=torch.int32)
    w = torch.rand(B, n, 3, device=DEV)
    w = w / w.sum(-1, keepdim=True)
    o16, o32 = _ext.three_interpolate(feats, iidx, w), _ext.three_interpolate(feats.float(), iidx, w)
    assert torch.equal(o16, o32.to(BF16))
    li = iidx.view(B, 1, -1).long().expand(B, 256, -1)
    want = (torch.gather(feats.double(), 2, li).view(B, 256, n, 3) * w.double()[:, None]).sum(-1)
    assert bool(((o16.double() - want).abs() <= _bf16_ulp(want).double() + 1e-6).all())
    gi = torch.randn(B, 256, n, device=DEV).to(BF16)
    t16, t32 = _ext.three_interpolate_grad(gi, iidx, w, m), _ext.three_interpolate_grad(gi.float(), iidx, w, m)
    assert bool(((t16.float() - t32).abs() <= _bf16_ulp(t32) + 1e-5 * t32.abs().max()).all())


# ---- module level ----------------------------------------------------------------------------------------------------------
DET_SCENES, DET_POINTS = 4, 20000
# bf16 against the fp32 step, relative: |loss_bf16 - loss_fp32| / |loss_fp32| and, per parameter,
# ||grad_bf16 - grad_fp32|| / ||grad_fp32||.  bf16 keeps 8 significant bits and every activation and incoming gradient
# is rounded once per layer, so the loss moves by ~1e-3 (9.4e-4 measured on a B200).  The BatchNorm bias and weight
# gradients of the early layers are sums of dm with heavy cancellation and move by up to 0.77 (measured); a dropped
# position partition of the bf16 list-based grouping backward raises that to 1.9, a bf16 BatchNorm backward without
# the sum(dm)/M term to 13.  Parameters whose fp32 gradient is below 1e-6 of the largest (biases of convolutions
# followed by a BatchNorm: zero up to rounding) carry no relative information and are left out.
REL_BAR_LOSS = 0.02
REL_BAR_GRAD = 1.0


def _amp():
    return torch.autocast("cuda", dtype=BF16, cache_enabled=False)


def _detector():
    from spacap3d_b200.detector import VoteNetDetector
    torch.manual_seed(0)
    return VoteNetDetector(input_feature_dim=1).to(DEV).train()


def _det_inputs():
    from spacap3d_b200.scenes import make_scene
    return torch.from_numpy(np.stack([make_scene(5000 + i, DET_POINTS) for i in range(DET_SCENES)], 0)).to(DEV)


def _det_loss(out):
    """Votes and their features: everything before the vote aggregation, whose FPS and ball query run on computed
    vote coordinates (a bf16 rounding can move a sample there, and with it everything downstream, by a discrete amount)."""
    return ((out["vote_xyz"].float() ** 2).sum() + (out["vote_features"].float() ** 2).sum()) * 1e-3


def _det_step(model, pc, amp):
    model.zero_grad(set_to_none=False)
    with (_amp() if amp else torch.autocast("cuda", enabled=False)):
        out = model({"point_clouds": pc})
        loss = _det_loss(out)
    loss.backward()
    return out, loss


def _det_result(model, out, loss):
    return dict(loss=float(loss.detach()), out={k: out[k].detach().float().clone() for k in ("vote_xyz", "vote_features", "center")},
                grads={n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None},
                running={n: b.detach().clone() for n, b in model.named_buffers() if "running" in n})


def _tf32_off():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False


def bf16_vs_fp32_errors():
    """(loss relative error, {parameter: gradient relative error}) of one bf16 autocast step against the fp32 step."""
    _tf32_off()
    pc = _det_inputs()
    res = []
    for amp in (False, True):
        model = _detector()
        out, loss = _det_step(model, pc, amp)
        res.append(_det_result(model, out, loss))
    a, b = res
    top = max(float(g.norm()) for g in a["grads"].values())
    grads = {n: float((b["grads"][n].float() - g).norm() / g.norm()) for n, g in a["grads"].items()
             if float(g.norm()) > 1e-6 * top}
    return abs(b["loss"] - a["loss"]) / abs(a["loss"]), grads


@pytest.fixture
def lib_calls(monkeypatch):
    from spacap3d_b200 import _lib
    names = []
    real = _lib.call

    def spy(name, *args):
        names.append(name)
        return real(name, *args)

    monkeypatch.setattr(_lib, "call", spy)
    return names


@pytest.mark.gpu
def test_detector_step_bf16_eager_graph_and_entry_points(lib_calls):
    """One autocast training step: the bf16 twins run for every fused BatchNorm layer (19: 4 SA x 3 + 2 FP x 2 +
    vote aggregation x 3) and for the grouping of SA2-SA4 and the vote aggregation; the same step captured in a CUDA
    graph and replayed from the same state gives bit-equal forward outputs and running statistics."""
    from spacap3d_b200 import pytorch_utils
    assert pytorch_utils.FUSED_BN_RELU_TRAINING
    torch.backends.cudnn.deterministic = True
    pc = _det_inputs()
    model = _detector()
    state = {k: v.clone() for k, v in model.state_dict().items()}
    n0 = len(lib_calls)
    eager = _det_result(model, *_det_step(model, pc, True))
    calls = lib_calls[n0:]
    fused_fwd = [c for c in calls if c.startswith("spc_bn_relu") and c.endswith("forward_bf16")]
    assert len(fused_fwd) == 19, calls
    assert not [c for c in calls if c.startswith("spc_bn_relu") and not c.endswith("_bf16")
                and c != "spc_bn_relu_workspace_bytes"], calls
    assert calls.count("spc_group_points_bf16") >= 4, calls       # features of SA2-SA4 and the vote aggregation
    assert any(c.startswith("spc_group_points_grad") and c.endswith("_bf16") for c in calls), calls
    assert "spc_three_interpolate_bf16" in calls and "spc_three_interpolate_grad_bf16" in calls, calls
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _det_step(model, pc, True)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out, loss = _det_step(model, pc, True)
    model.load_state_dict(state)
    graph.replay()
    torch.cuda.synchronize()
    graphed = _det_result(model, out, loss)
    for k in eager["out"]:
        assert torch.equal(graphed["out"][k], eager["out"][k]), k
    for n in eager["running"]:
        assert torch.equal(graphed["running"][n], eager["running"][n]), n
    assert set(graphed["grads"]) == set(eager["grads"])
    torch.backends.cudnn.deterministic = False


@pytest.mark.gpu
def test_detector_step_bf16_against_fp32():
    """Loss within REL_BAR_LOSS and every parameter gradient within REL_BAR_GRAD of the fp32 step (relative).  A
    dropped position partition of the bf16 list-based grouping backward, or a bf16 BatchNorm backward without the
    sum(dm)/M term, exceeds these bars."""
    loss_err, grads = bf16_vs_fp32_errors()
    assert loss_err < REL_BAR_LOSS, loss_err
    worst = max(grads, key=grads.get)
    assert grads[worst] < REL_BAR_GRAD, (worst, grads[worst])


@pytest.mark.gpu
def test_detector_step_bf16_with_torch_batchnorm():
    """FUSED_BN_RELU_TRAINING = False: torch's BatchNorm in bf16, the grouping and interpolation twins still run."""
    from spacap3d_b200 import pytorch_utils
    pytorch_utils.FUSED_BN_RELU_TRAINING = False
    try:
        model = _detector()
        out, loss = _det_step(model, _det_inputs(), True)
        assert torch.isfinite(loss) and all(bool(torch.isfinite(p.grad).all()) for p in model.parameters()
                                            if p.grad is not None)
    finally:
        pytorch_utils.FUSED_BN_RELU_TRAINING = True


@pytest.mark.gpu
def test_fp32_step_calls_no_bf16_entry_point(lib_calls):
    """Without autocast the training step calls only the entry points that existed before the bf16 twins."""
    from spacap3d_b200 import _lib
    model = _detector()
    _det_step(model, _det_inputs(), False)
    parent = set(_lib.SIGNATURES) - {n + "_bf16" for n in _lib.BF16_TWINS}
    assert lib_calls and set(lib_calls) <= parent, sorted(set(lib_calls) - parent)
