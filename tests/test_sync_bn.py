"""Synchronised BatchNorm in the fused training kernels: nn.SyncBatchNorm.convert_sync_batchnorm on a model of this
package makes every fused BatchNorm + ReLU (+ max-pool) block normalise with the statistics of all ranks.

  * Kernel level (one process): 2 and 3 ranks are emulated by filling the exchange rows of each rank by hand and
    summing them, which is what the SUM all-reduce does.  Every rank's slice is built from whole blocks of the dyadic
    generator of test_exact_training_kernels.py, so each rank's mean and M2 and their rank-order combination are
    exact, and the outputs are compared by torch.equal with the float64 evaluation over the concatenated batch, with
    that file's two exceptions (running_var within one ulp; dy within its bound when the global count is not a power
    of two).
  * Module level: two processes on one GPU (gloo) against one process on the whole batch, and without conversion as
    the negative control.
  * Paths that must not change: plain BatchNorm2d, a converted model without a process group, eval.
  * Whole detector on two GPUs (NCCL), eager and captured in a CUDA graph; skipped on a machine with one GPU.
"""
import datetime
import functools
import math
import os
import queue
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn

from test_exact_training_kernels import (BN_MOMENTUM, DEV, _BLOCK, _bn_reference, _check_bn_outputs, _expect_equal,
                                         _gen, _ints, _poison, make_bn)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K = 3                                   # values per channel in an exchanged row (SPC_BN_SYNC_K)

# ---- kernel level ---------------------------------------------------------------------------------------------------
# ranks: local batch sizes (0 = an empty shard); rest: the dimensions after C.  Every rank's B_r * prod(rest) is a
# multiple of 16.  d / p (default 0 / 1): rank r's slice is mu + a * (d_r + p_r * t), so its mean is mu + d_r a and its
# variance (p_r a)^2.  With different d_r the rank-order merge has to weight the means by the counts and add the
# between-rank term d^2 n nb / nn; the cases that use it have count ratios that keep every step of the merge dyadic
# (nb / nn in {1, 1/2, 1/4, 3/4}) and a global variance of 4 a^2, so every statistic stays exact.
SYNC_CASES = [
    dict(id="2r-vec-pow2", ranks=(2, 2), C=8, rest=(1024,)),                  # M = 4096: dy exact
    dict(id="3r-vec-pow2", ranks=(1, 1, 2), C=6, rest=(512,)),
    dict(id="2r-uneven-3+2", ranks=(3, 2), C=7, rest=(1024,)),                # M = 5120: dy bounded
    dict(id="3r-scalar-S6", ranks=(24, 16, 8), C=5, rest=(6,)),              # S % 4 != 0: the scalar kernels
    dict(id="2r-BC80000-slices", ranks=(2, 1), C=40000, rest=(16,)),         # B*C > 65535 on rank 0
    dict(id="2r-1+3-means", ranks=(1, 3), C=8, rest=(1024,), d=(-3, 1)),     # counts 1:3, means apart by 4a
    dict(id="2r-3+1-means-scales-scalar", ranks=(24, 8), C=5, rest=(6,), d=(-4, -2), p=(2, 1)),   # M = 192
    dict(id="3r-1+1+2-means-scales", ranks=(1, 1, 2), C=6, rest=(512,), d=(-4, -4, -1), p=(1, 2, 1)),
    dict(id="2r-empty-rank", ranks=(0, 2), C=8, rest=(512,)),                 # rank 0 holds no scene
]
SYNC_POOL_CASES = [
    dict(id="2r-ns16-pow2", ranks=(2, 2), C=6, rest=(64, 16)),
    dict(id="2r-ns32-uneven-3+2", ranks=(3, 2), C=5, rest=(100, 32)),
    dict(id="3r-ns64-uneven", ranks=(1, 2, 1), C=4, rest=(48, 64)),
    dict(id="2r-ns16-BC66000-slices", ranks=(2, 2), C=33000, rest=(4, 16)),
    dict(id="2r-ns16-1+3-means", ranks=(1, 3), C=6, rest=(64, 16), d=(-3, 1)),
    dict(id="3r-ns32-1+1+2-means-scales", ranks=(1, 1, 2), C=5, rest=(100, 32), d=(-4, -4, -1), p=(2, 1, 1)),
    dict(id="3r-ns16-empty-rank", ranks=(2, 0, 1), C=4, rest=(64, 16)),
]


def _offsets(c):
    R = len(c["ranks"])
    return c.get("d", (0,) * R), c.get("p", (1,) * R)


def make_sync_bn(c, pool):
    """make_bn over the concatenated batch for gamma, beta, dz and the running buffers, with y replaced by one built
    rank by rank: slice r is mu + a * (d_r + p_r * t) with t made of whole blocks (mean 0, variance 1) and t = 0 at
    the slice's first element, so that rank r's mean is mu + d_r a, its M2 is M_r (p_r a)^2 and the kernel's shift K
    is its mean.  Returns (operands, per-rank means, per-rank M2)."""
    C, rest = c["C"], c["rest"]
    S = math.prod(rest)
    B = sum(c["ranks"])
    dev = "cpu" if B * C * S <= 2 ** 22 else DEV
    d = make_bn(dict(id=c["id"], shape=(B, C) + rest), dev, pool=pool)
    g = _gen(c["id"] + "/ranks", dev)
    a = 2.0 ** _ints(-3, 2, (C,), g, dev)
    mu = _ints(-64, 64, (C,), g, dev) / 16
    ys, means, m2s = [], [], []
    for br, dr, pr in zip(c["ranks"], *_offsets(c)):
        M_r = br * S
        assert M_r % len(_BLOCK) == 0
        means.append(mu + dr * a if br else torch.zeros_like(mu))
        m2s.append(M_r * (pr * a) ** 2)
        if not br:
            continue
        t = torch.tensor(_BLOCK, dtype=torch.float32, device=dev)[
            torch.argsort(torch.rand(C, M_r, generator=g, device=dev), dim=1) % len(_BLOCK)]
        first0 = (t == 0).to(torch.uint8).argmax(1)
        rows = torch.arange(C, device=dev)
        t[rows, first0] = t[:, 0].clone()
        t[:, 0] = 0
        yr = mu[:, None] + a[:, None] * (dr + pr * t.double())
        ys.append(yr.view(C, br, S).transpose(0, 1).reshape((br, C) + rest))
    d["y"] = torch.cat(ys, 0)
    return d, means, m2s


def _slices(ranks):
    b, out = 0, []
    for br in ranks:
        out.append(slice(b, b + br))
        b += br
    return out


def _local_sums(d, ref, sl, pool):
    """(dbeta, dgamma) of one rank: sums of dm and dm * xhat over its slice, with the global statistics."""
    y, dz = d["y"][sl], d["dz"][sl]
    red = tuple(i for i in range(y.dim()) if i != 1)
    bc = lambda v: v.view((1, -1) + (1,) * (y.dim() - 2))          # noqa: E731
    xh = (y - bc(ref["mean"])) * bc(ref["invstd"])
    zp = bc(d["gamma"]) * xh + bc(d["beta"])
    if pool:
        am = ref["argmax"][sl].unsqueeze(-1)
        dm = torch.zeros_like(y).scatter_(-1, am, torch.where(zp.gather(-1, am) > 0, dz[..., None], 0.0))
    else:
        dm = torch.where(zp > 0, dz, 0.0)
    return dm.sum(red), (dm * xh).sum(red)


def _run_sync_case(c, pool):
    from spacap3d_b200 import _ext
    d, means, m2s = make_sync_bn(c, pool)
    ref = _bn_reference(d, pool=pool)
    C, ranks = c["C"], c["ranks"]
    R = len(ranks)
    sls = _slices(ranks)
    f = lambda k: d[k].float().to(DEV)                              # noqa: E731
    y, gamma, beta, dz = f("y"), f("gamma"), f("beta"), f("dz")
    # forward: each rank fills its row of its own zeroed buffer; the all-reduce is their sum
    bufs = []
    for r, sl in enumerate(sls):
        buf = torch.zeros(R, C, K, dtype=torch.float64, device=DEV)
        _ext.bn_relu_sync_stats(y[sl].contiguous(), buf[r])
        bufs.append(buf)
    rows = sum(bufs)
    for r, sl in enumerate(sls):
        M_r = ranks[r] * math.prod(c["rest"])
        _expect_equal(rows[r, :, 0], torch.full((C,), float(M_r), dtype=torch.float64, device=DEV), "row %d n" % r)
        _expect_equal(rows[r, :, 1], means[r].to(DEV), "row %d mean" % r)
        _expect_equal(rows[r, :, 2], m2s[r].to(DEV), "row %d M2" % r)
    outs, saved = [], []
    for r, sl in enumerate(sls):
        yr = y[sl].contiguous()
        rm, rv = f("rm"), f("rv")
        _poison(yr.shape)
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
    for r in range(1, R):                         # identical statistics and running buffers on every rank
        for k in ("mean", "invstd", "rm", "rv"):
            assert torch.equal(outs[r][k], outs[0][k]), (c["id"], r, k)
    # backward: local dgamma / dbeta, then the exchanged sums
    bufs, local = [], []
    for r, sl in enumerate(sls):
        yr, mean, invstd = saved[r]
        buf = torch.zeros(R, C, K, dtype=torch.float64, device=DEV)
        dzr = dz[sl].contiguous()
        if pool:
            dgamma, dbeta = _ext.bn_relu_maxpool_sync_backward_reduce(dzr, outs[r]["ymax"], yr, gamma, beta, mean,
                                                                      invstd, buf[r])
        else:
            dgamma, dbeta = _ext.bn_relu_sync_backward_reduce(dzr, yr, gamma, beta, mean, invstd, buf[r])
        bufs.append(buf)
        local.append((dgamma, dbeta))
    rows = sum(bufs)
    for r, sl in enumerate(sls):
        yr, mean, invstd = saved[r]
        dzr = dz[sl].contiguous()
        _poison(yr.shape)
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
        _check_bn_outputs(rref, dict(outs[r], dy=dy, dgamma=local[r][0], dbeta=local[r][1]),
                          "%s rank %d" % (c["id"], r))


@pytest.mark.gpu
@pytest.mark.parametrize("c", SYNC_CASES, ids=[c["id"] for c in SYNC_CASES])
def test_bn_relu_sync_exact(c):
    """The plain synced entry points: z, mean, invstd, running_mean, local dgamma / dbeta bit for bit on every rank,
    running_var within one ulp, dy bit for bit (global count a power of two) or within its bound."""
    _run_sync_case(c, pool=False)


@pytest.mark.gpu
@pytest.mark.parametrize("c", SYNC_POOL_CASES, ids=[c["id"] for c in SYNC_POOL_CASES])
def test_bn_relu_maxpool_sync_exact(c):
    """The max-pool synced entry points: pooled, the winning slot, the pre-BN value there and everything above."""
    _run_sync_case(c, pool=True)


def test_sync_cases_meet_preconditions():
    """Every rank's slice is whole generator blocks, the cases reach both dy regimes, the scalar path and a local
    B*C above the 65535 rows of one launch."""
    pow2, other = False, False
    for pool, cases in ((False, SYNC_CASES), (True, SYNC_POOL_CASES)):
        for c in cases:
            S = math.prod(c["rest"])
            assert all(br * S % len(_BLOCK) == 0 for br in c["ranks"]), c["id"]
            M = sum(c["ranks"]) * S
            assert M < 2 ** 22
            pow2 |= M & (M - 1) == 0
            other |= M & (M - 1) != 0
            if pool:
                assert c["rest"][1] in (16, 32, 64)
    assert pow2 and other
    assert any(c["rest"][-1] % 4 for c in SYNC_CASES)
    assert any(max(c["ranks"]) * c["C"] > 65535 for c in SYNC_CASES)
    assert any(max(c["ranks"]) * c["C"] > 65535 for c in SYNC_POOL_CASES)
    assert any(len(set(c["ranks"])) > 1 for c in SYNC_CASES + SYNC_POOL_CASES)
    for cases in (SYNC_CASES, SYNC_POOL_CASES):
        assert any(len(set(_offsets(c)[0])) > 1 and len(set(c["ranks"])) > 1 for c in cases)   # counts weigh means
        assert any(len(set(_offsets(c)[1])) > 1 for c in cases)
        assert any(0 in c["ranks"] for c in cases)
    for c in SYNC_CASES + SYNC_POOL_CASES:
        n, mean, m2 = _rank_order_merge(c)
        var = m2 / n                                       # in units of a^2: invstd = 1 / (sqrt(var) a) exact
        while var >= 4:
            var /= 4
        assert var == 1, (c["id"], m2 / n)


def _dyadic(x):
    return x.denominator & (x.denominator - 1) == 0


def _rank_order_merge(c):
    """bn_sync_finalize_forward_kernel's merge in exact rationals (units of a), asserting that every quantity it
    forms is dyadic with few bits, i.e. exact in float64."""
    from fractions import Fraction
    S = math.prod(c["rest"])
    n, mean, m2 = Fraction(0), Fraction(0), Fraction(0)
    for br, dr, pr in zip(c["ranks"], *_offsets(c)):
        nb = Fraction(br * S)
        if not nb:
            continue
        nn = n + nb
        dd = dr - mean
        if dd:                          # with equal means the weights are rounded but multiply an exact zero
            for x in (nb / nn, n * nb / nn, dd * (nb / nn), dd * dd * (n * nb / nn)):
                assert _dyadic(x) and abs(x.numerator) < 2 ** 40, (c["id"], x)
        mean, m2, n = mean + dd * (nb / nn), m2 + nb * pr * pr + dd * dd * (n * nb / nn), nn
    return n, mean, m2


# ---- module level ---------------------------------------------------------------------------------------------------
N_SCENES, N_POINTS = 4, 3000


def _stack(dev):
    from spacap3d_b200.pointnet2_modules import PointnetFPModule, PointnetSAModuleVotes
    torch.manual_seed(7)
    sa1 = PointnetSAModuleVotes(npoint=256, radius=0.4, nsample=16, mlp=[4, 32, 32, 64], use_xyz=True,
                                normalize_xyz=True)
    sa2 = PointnetSAModuleVotes(npoint=64, radius=0.8, nsample=16, mlp=[64, 64, 64, 128], use_xyz=True,
                                normalize_xyz=True)
    fp = PointnetFPModule(mlp=[128 + 64, 64, 64])
    return torch.nn.ModuleList([sa1, sa2, fp]).to(dev).train()


def _inputs(total=N_SCENES):
    from spacap3d_b200.scenes import make_scene_xyz
    xyz = torch.from_numpy(np.stack([make_scene_xyz(90 + i, N_POINTS) for i in range(total)], 0))
    feats = torch.randn(total, 4, N_POINTS, generator=torch.Generator().manual_seed(2))
    return xyz, feats


def _stack_step(model, xyz, feats, dev):
    """Forward + backward of a loss that is a sum over scenes; returns everything compared, on the CPU."""
    xyz = xyz.to(dev).requires_grad_(True)
    feats = feats.to(dev).requires_grad_(True)
    sa1, sa2, fp = model
    x1, f1, _ = sa1(xyz, feats)
    x2, f2, _ = sa2(x1, f1)
    up = fp(x1, x2, f1, f2)
    loss = ((up ** 2).sum() + (f2 ** 2).sum() + x2.sum()) * 1e-3
    loss.backward()
    return dict(up=up.detach().cpu(), f2=f2.detach().cpu(), dxyz=xyz.grad.cpu(), dfeats=feats.grad.cpu(),
                grads=[p.grad.cpu() for p in model.parameters()],
                running=[b.cpu() for n, b in model.named_buffers() if "running" in n])


def _tf32_off():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _module_worker(rank, world, port, q, total=N_SCENES):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        sys.path.insert(0, ROOT)
        import torch.distributed as dist
        dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=120))
        from spacap3d_b200.dist import shard_range
        _tf32_off()
        dev = torch.device("cuda", 0)
        xyz, feats = _inputs(total)
        b, e = shard_range(total, rank, world)
        res = {}
        for convert in (True, False):
            model = _stack(dev)
            if convert:
                model = nn.SyncBatchNorm.convert_sync_batchnorm(model)
            res[convert] = _stack_step(model, xyz[b:e], feats[b:e], dev)
        q.put((rank, _to_numpy(res)))
        dist.barrier()
        dist.destroy_process_group()
    except BaseException as exc:           # report instead of leaving the parent waiting
        q.put((rank, repr(exc)))
        raise


def _to_numpy(obj):
    """Results cross the process boundary by value (the sending rank may have exited before they are read)."""
    if isinstance(obj, torch.Tensor):
        return obj.numpy()
    if isinstance(obj, dict):
        return {k: _to_numpy(v) for k, v in obj.items()}
    if isinstance(obj, list):
        return [_to_numpy(v) for v in obj]
    return obj


def _to_torch(obj):
    if isinstance(obj, np.ndarray):
        return torch.from_numpy(obj)
    if isinstance(obj, dict):
        return {k: _to_torch(v) for k, v in obj.items()}
    if isinstance(obj, list):
        return [_to_torch(v) for v in obj]
    return obj


def _spawn(target, world, timeout):
    """Run target(rank, world, port, q) in `world` spawned processes; their results by rank.  Children that do not
    finish in time are killed, so a mismatch fails the test instead of hanging it."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000) + 7
    procs = [ctx.Process(target=target, args=(r, world, port, q)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        res = {}
        for _ in procs:
            try:
                rank, val = q.get(timeout=timeout)
            except queue.Empty:
                pytest.fail("a rank did not report within %d s" % timeout)
            assert not isinstance(val, str), "rank %d failed: %s" % (rank, val)
            res[rank] = _to_torch(val)
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
        return [res[r] for r in range(world)]
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join(timeout=10)


def _close(a, b, grad):
    """Gradients and running statistics: the tolerance of tests/test_training_gpu.py.  Forward outputs: the tolerance
    tests/test_bn_relu_gpu.py uses for the fused against the unfused BatchNorm, because here too the statistics are
    summed in another order (per rank, then merged) and, in addition, the convolutions run on half batches."""
    if grad:
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-5 * max(1.0, b.abs().max().item()))
    else:
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-5)


def _compare_sharded(parts, full, slices):
    """Per-rank outputs and input gradients against their slice of the single-process run, the sum of the ranks'
    parameter gradients against its gradients, every rank's running statistics against its buffers.  Raises one
    AssertionError naming every mismatch."""
    bad = []

    def check(what, a, b, grad):
        try:
            _close(a, b, grad)
        except AssertionError as e:
            bad.append("%s: %s" % (what, str(e).replace("\n", " ")))

    for r, (part, sl) in enumerate(zip(parts, slices)):
        for k in ("up", "f2"):
            check("rank %d %s" % (r, k), part[k], full[k][sl], grad=False)
        for k in ("dxyz", "dfeats"):
            check("rank %d %s" % (r, k), part[k], full[k][sl], grad=True)
        for i, (a, b) in enumerate(zip(part["running"], full["running"])):
            check("rank %d running buffer %d" % (r, i), a, b, grad=True)
    for i, b in enumerate(full["grads"]):
        check("parameter gradient %d" % i, sum(p["grads"][i] for p in parts), b, grad=True)
    if bad:
        raise AssertionError("\n".join(bad))


@pytest.mark.gpu
def test_two_ranks_match_one_process():
    """SA (nsample 16: the fused max-pool) -> SA -> FP, every block with BatchNorm, converted, in training: two ranks
    with two scenes each equal one process with all four; the unconverted two-rank run does not."""
    _two_ranks_against_one_process(4)


@pytest.mark.gpu
def test_two_uneven_ranks_match_one_process():
    """The same with three scenes, two on rank 0 and one on rank 1: the exchanged counts weigh the ranks."""
    _two_ranks_against_one_process(3)


def _two_ranks_against_one_process(total):
    from spacap3d_b200.dist import shard_range
    parts = _spawn(functools.partial(_module_worker, total=total), 2, timeout=600)
    _tf32_off()
    xyz, feats = _inputs(total)
    full = _stack_step(_stack(DEV), xyz, feats, DEV)
    slices = [slice(*shard_range(total, r, 2)) for r in range(2)]
    _compare_sharded([p[True] for p in parts], full, slices)
    for a, b in zip(parts[0][True]["running"], parts[1][True]["running"]):
        assert torch.equal(a, b)                                   # bit-equal across ranks
    with pytest.raises(AssertionError):                           # negative control: per-rank statistics
        _compare_sharded([p[False] for p in parts], full, slices)


# ---- paths that must not change -------------------------------------------------------------------------------------
def test_sync_group_only_with_a_process_group():
    """Without an initialised process group a SyncBatchNorm takes the unsynchronised path, like torch's own."""
    from spacap3d_b200.pytorch_utils import _sync_group
    assert _sync_group(nn.BatchNorm2d(4)) is None
    assert _sync_group(nn.SyncBatchNorm(4)) is None


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
@pytest.mark.parametrize("mode", ["batchnorm2d", "converted-no-group", "eval"])
def test_unsynchronised_paths_unchanged(mode, lib_calls):
    """No synced entry point runs for plain BatchNorm2d, for a converted model without a process group, or in eval.
    In the last two the converted model makes the same library calls as the unconverted one, and its forward outputs
    and running statistics are bit-equal.  Its gradients are compared within the tolerance of test_training_gpu.py:
    they pass through atomic scatter-adds (grouping of 3- and 4-channel inputs), whose order varies between runs."""
    _tf32_off()
    xyz, feats = _inputs()
    xyz, feats = xyz[:2], feats[:2]
    runs, calls = [], []
    for convert in (False, True):
        model = _stack(DEV)
        if convert:
            model = nn.SyncBatchNorm.convert_sync_batchnorm(model)
            assert any(isinstance(m, nn.SyncBatchNorm) for m in model.modules())
        first = len(lib_calls)
        if mode == "eval":
            model.eval()
            with torch.no_grad():
                sa1, sa2, fp = model
                x1, f1, _ = sa1(xyz.to(DEV), feats.to(DEV))
                x2, f2, _ = sa2(x1, f1)
                runs.append(dict(up=fp(x1, x2, f1, f2).cpu(), f2=f2.cpu()))
        else:
            runs.append(_stack_step(model, xyz, feats, DEV))
        calls.append(lib_calls[first:])
        if mode == "batchnorm2d":
            break
    assert lib_calls and not [n for n in lib_calls if "_sync" in n], sorted(set(lib_calls))
    if mode == "batchnorm2d":
        assert "spc_bn_relu_maxpool_train_forward" in lib_calls and "spc_bn_relu_train_backward" in lib_calls
        return
    assert calls[0] == calls[1]
    a, b = runs
    for k in ("up", "f2"):
        assert torch.equal(a[k], b[k]), k
    if mode == "eval":
        return
    assert all(torch.equal(u, v) for u, v in zip(a["running"], b["running"]))
    for u, v in zip([a["dxyz"], a["dfeats"]] + a["grads"], [b["dxyz"], b["dfeats"]] + b["grads"]):
        _close(u, v, grad=True)


# ---- whole detector, two GPUs, NCCL ---------------------------------------------------------------------------------
DET_SCENES, DET_POINTS = 4, 20000


def _detector(dev, convert):
    from spacap3d_b200.detector import VoteNetDetector
    torch.manual_seed(0)
    model = VoteNetDetector(input_feature_dim=1).to(dev).train()
    return nn.SyncBatchNorm.convert_sync_batchnorm(model) if convert else model


def _det_inputs():
    from spacap3d_b200.scenes import make_scene
    return torch.from_numpy(np.stack([make_scene(5000 + i, DET_POINTS) for i in range(DET_SCENES)], 0))


def _det_loss(out):
    """A sum over scenes of the votes and their features.  Everything before the vote aggregation: its FPS and ball
    query run on computed vote coordinates, so an fp32 rounding difference between a 2 x 2 and a 1 x 4 run can change
    a sample there and with it everything downstream by a large, discrete amount.  The proposal head still runs its
    forward (and its SyncBatchNorm collectives) but receives no gradient."""
    return ((out["vote_xyz"] ** 2).sum() + (out["vote_features"] ** 2).sum()) * 1e-3


def _det_step(model, pc):
    model.zero_grad(set_to_none=False)
    out = model({"point_clouds": pc})
    _det_loss(out).backward()
    return out


def _det_result(model, out):
    return dict(out={k: out[k].detach().cpu().clone() for k in ("vote_xyz", "vote_features", "center")},
                grads={n: p.grad.detach().cpu().clone() for n, p in model.named_parameters() if p.grad is not None},
                running={n: b.detach().cpu().clone() for n, b in model.named_buffers() if "running" in n})


def _detector_worker(rank, world, port, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        sys.path.insert(0, ROOT)
        import torch.distributed as dist
        from spacap3d_b200.dist import shard_range
        dev = torch.device("cuda", rank)
        torch.cuda.set_device(dev)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev,
                                timeout=datetime.timedelta(seconds=180))
        _tf32_off()
        torch.backends.cudnn.deterministic = True          # eager and replay must take the same cuDNN algorithms
        b, e = shard_range(DET_SCENES, rank, world)
        pc = _det_inputs()[b:e].to(dev)
        model = _detector(dev, True)
        state = {k: v.clone() for k, v in model.state_dict().items()}
        eager = _det_result(model, _det_step(model, pc))
        # the same step captured in a CUDA graph (warmed up on a side stream), replayed from the same state
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            _det_step(model, pc)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = _det_step(model, pc)
        model.load_state_dict(state)
        graph.replay()
        torch.cuda.synchronize()
        q.put((rank, _to_numpy(dict(eager=eager, graphed=_det_result(model, out)))))
        dist.barrier()
        dist.destroy_process_group()
    except BaseException as exc:
        q.put((rank, repr(exc)))
        raise


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_detector_two_gpus_nccl():
    """Whole detector, converted, one training step: 2 ranks x 2 scenes against 1 process x 4 scenes up to the vote
    aggregation (see _det_loss), running statistics bit-equal across ranks, and the same step captured in a CUDA graph
    equal to its eager run when replayed: forward outputs and running statistics bit for bit, gradients within the
    tolerance of test_training_gpu.py (they pass through atomic scatter-adds, whose order varies between runs)."""
    from spacap3d_b200.dist import shard_range
    parts = _spawn(_detector_worker, 2, timeout=900)
    _tf32_off()
    model = _detector(DEV, False)
    full = _det_result(model, _det_step(model, _det_inputs().to(DEV)))
    before_aggregation = [n for n in full["running"] if not n.startswith("proposal.")]
    assert before_aggregation and set(full["grads"]) and not any(n.startswith("proposal.") for n in full["grads"])
    for r, p in enumerate(parts):
        eager, graphed = p["eager"], p["graphed"]
        sl = slice(*shard_range(DET_SCENES, r, 2))
        for k in ("vote_xyz", "vote_features"):
            _close(eager["out"][k], full["out"][k][sl], grad=False)
        for n in before_aggregation:
            _close(eager["running"][n], full["running"][n], grad=True)
        for k in eager["out"]:
            assert torch.equal(graphed["out"][k], eager["out"][k]), (r, k)
        for n in eager["running"]:
            assert torch.equal(graphed["running"][n], eager["running"][n]), (r, n)
        assert set(graphed["grads"]) == set(eager["grads"]) == set(full["grads"])
        for n in eager["grads"]:
            _close(graphed["grads"][n], eager["grads"][n], grad=True)
    for n in full["running"]:
        assert torch.equal(parts[0]["eager"]["running"][n], parts[1]["eager"]["running"][n]), n
    for n, b in full["grads"].items():
        _close(parts[0]["eager"]["grads"][n] + parts[1]["eager"]["grads"][n], b, grad=True)
