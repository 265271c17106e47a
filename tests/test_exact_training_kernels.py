"""The training path's scatter, interpolation and BatchNorm kernels bit for bit, on data where no rounding happens.

Every training step runs the backward passes of grouping and sampling (csrc/group.cu), three_interpolate and its
backward (csrc/interp.cu) and the training-mode BatchNorm + ReLU kernels, with and without the fused max-pool
(csrc/bn_relu.cu).  Which kernel, which template instantiation and which tiling runs is chosen from the shapes, and the
training sweep (4 scenes per GPU at 1-5x the SA npoints) crosses thresholds that the tolerance tests of
test_ops_gpu.py and test_bn_relu_gpu.py never reach.  Here every input lies on a dyadic grid with so few significant
bits that every product and every partial sum is exact in fp32, in any order and under any partitioning, so each
output has exactly one correct value, the float64 evaluation with plain torch ops on the device, and the kernels are
compared with it by torch.equal:

  * scatters (group_points_grad, gather_points_grad): gradients k/8, |k| <= 8.  An output sums at most S terms, so
    S * 8 < 2^24 keeps every partial sum exact; the bound is taken from S, not from the drawn data.
  * three_interpolate: points and gradients k/8 in [-1, 1], weights k/16 in [0, 1] (zero weights, repeated indices,
    rows that do not sum to 1).  Products sit on the grid 2^-7; the backward sums at most 3n of them: 3n * 2^7 < 2^24.
  * BatchNorm: per channel y = mu + a * t with mu a multiple of 2^-4, a = 2^e and t a random arrangement of blocks of
    sixteen values {-2, 2, -1 x4, 1 x4, 0 x6}, t = 0 at (b=0, s=0) so that the kernel's shift K is mu.  Then the batch
    mean is mu, the biased variance a^2 and invstd 1/a (or 1/(2a) with eps = 3a^2), all exact; the sums of the
    statistics pass stay below 2^24 units while M = B*S < 2^22.  gamma = +-2^k, beta is either -gamma * xhat(t0)
    for a t0 of the channel (z = 0 occurs exactly: the ReLU convention "gradient only where the output is > 0" is
    tested, not masked) or k/8, or puts every z of the channel at or below 0.  dz in {0, +-1/2, +-1}, or {0, +-1}
    for the large cases, where dy's intermediates would not fit 24 bits on the finer grid.

Where exactness stops: running_var scales by M/(M-1) (compared within one fp32 ulp), and when M is not a power of two
inv_M = fl(1/M) rounds, so dy is held to the bound derived in _bn_reference from its fp32 operations; every other
output stays exact.  Whether dy's intermediates fit 24 bits also depends on the draw when M is a power of two, so the
reference asserts it on the data it is given, on the CPU for small cases and on the device for the large ones.

The CPU-only tests check every precondition above for every case (large ones analytically from their generator
parameters) and, with a restatement of the launch plans whose constants are read from the .cu sources, that every
branch of the plan functions named in BRANCHES is reached by some case.
"""
import math
import os
import re
import zlib

import numpy as np
import pytest
import torch

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "spacap3d_b200", "csrc")
FP32_UNITS = 2 ** 24           # an fp32 sum is exact while its magnitude stays below 2^24 units of its grid


# ---- launch-plan constants, read from the sources ----------------------------------------------------------------
def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _num(expr):
    """'200 * 1024' -> 204800."""
    return math.prod(int(x) for x in expr.split("*"))


def _constants():
    src = {n: _read(n) for n in ("group.cu", "interp.cu", "bn_relu.cu", "common.cuh")}
    pats = {
        # name: (file, regex whose group 1 is the value)
        "kNumSMs": ("common.cuh", r"constexpr int kNumSMs = (\d+);"),
        "GP_ROW_BUDGET": ("group.cu", r"const size_t budget = ([\d *]+);"),
        "GP_CT_BYTES": ("group.cu", r"int ct = \(int\)\(\(([\d *]+)\) / row\);"),
        "GP_CT_MAX": ("group.cu", r"if \(ct > (\d+)\) ct = \d+;"),
        "GP_WAVES": ("group.cu", r"const long long want = (\d+)LL \* kNumSMs;"),
        "GP_CHUNK_MIN": ("group.cu", r"S / \(nchunks \* 2\) >= (\d+)"),
        "GG_PART_MAX": ("group.cu", r"constexpr int GG_PART_MAX = (\d+);"),
        "GG_CT_MAX": ("group.cu", r"constexpr int GG_CT_MAX = (\d+);"),
        "GG_SHORT": ("group.cu", r"constexpr int GG_SHORT = (\d+);"),
        "GG_CT_BYTES": ("group.cu", r"int ct = \(int\)\(\(([\d *]+)\) / \(\(size_t\)g\.Sp"),
        "GG_LISTS_SMEM": ("group.cu", r"g\.lists_smem = rows \+ lists <= ([\d *]+);"),
        "GB_MAX_N": ("group.cu", r"constexpr int GB_MAX_N = (\d+);"),
        "GL_CT": ("group.cu", r"constexpr int GL_CT = (\d+);"),
        "GL_LONG": ("group.cu", r"constexpr int GL_LONG = (\d+);"),
        "EX_MIN_C": ("group.cu", r"\(workspace\) & 15\) \|\| C < (\d+) \|\|"),
        "EX_POINTS_PER_C": ("group.cu", r"\(long long\)N > (\d+)LL \* C\)"),
        "TI_THREADS": ("interp.cu", r"constexpr int TI_THREADS = (\d+);"),
        "TI_CT": ("interp.cu", r"constexpr int TI_CT = (\d+);"),
        "TI_FWD_BYTES": ("interp.cu", r"\(int\)\(\(([\d *]+)\) / \(\(size_t\)m \* sizeof\(float\)\)\)"),
        "TI_FWD_CT_MAX": ("interp.cu", r"if \(CT > (\d+)\) CT = \d+;"),
        "TI_FWD_CT_MIN": ("interp.cu", r"while \(CT > (\d+) &&"),
        "TI_FWD_WAVES": ("interp.cu", r"< (\d+) \* kNumSMs\) CT /= 2;"),
        "TI_GRAD_OPTIN": ("interp.cu",
                          r"if \(smem > ([\d *]+)\)\s*SPC_CUDA\(cudaFuncSetAttribute\(three_interpolate_grad"),
        "TI_GRAD_SMEM_MAX": ("interp.cu", r"if \(smem <= ([\d *]+)\) \{"),
        "BN_THREADS": ("bn_relu.cu", r"constexpr int BN_THREADS = (\d+);"),
        "BN_MAX_SPLITS": ("bn_relu.cu", r"constexpr int BN_MAX_SPLITS = (\d+);"),
        "BN_CTAS_PER_SM": ("bn_relu.cu", r"int splits = ceil_div\((\d+) \* kNumSMs, C\);"),
        "BP_UNR": ("bn_relu.cu", r"constexpr int BP_UNR = (\d+);"),
        "BN_SLICE_ROWS": ("bn_relu.cu", r"static int sync_batch_slice\(int C\) \{ return max\(1, (\d+) / C\); \}"),
    }
    k = {}
    for name, (f, pat) in pats.items():
        m = re.search(pat, src[f])
        assert m, "constant %s not found in %s: the plan restatement below is stale" % (name, f)
        k[name] = _num(m.group(1))
    return k


def _cdiv(a, b):
    return -(-a // b)


# ---- restatement of the plan functions ---------------------------------------------------------------------------
def plan_group(K, B, C, N, S):
    """group.cu plan_group: (staged, CT, nchunks)."""
    row = 4 * N
    staged = row <= K["GP_ROW_BUDGET"] and N > 0
    CT = max(1, min(K["GP_CT_BYTES"] // row, C, K["GP_CT_MAX"])) if staged else 4
    ctiles = _cdiv(C, CT)
    nchunks = 1
    while B * ctiles * nchunks < K["GP_WAVES"] * K["kNumSMs"] and S // (nchunks * 2) >= K["GP_CHUNK_MIN"]:
        nchunks *= 2
    chunk = (_cdiv(S, nchunks) + 3) & ~3
    return staged, CT, _cdiv(S, chunk)


def plan_group_grad(K, C, N, S):
    """group.cu plan_group_grad: (H, Sp, CT, lists_smem)."""
    H = _cdiv(S, K["GG_PART_MAX"])
    Sp = _cdiv(_cdiv(S, H), 8) * 8
    H = _cdiv(S, Sp)
    Np = (N + 1 + 3) // 4 * 4
    CT = max(1, min(K["GG_CT_BYTES"] // (Sp * 4), K["GG_CT_MAX"], C))
    return H, Sp, CT, CT * Sp * 4 + Sp * 2 + Np * 4 <= K["GG_LISTS_SMEM"]


def grad_route(K, C, N, workspace):
    """Which kernel family spc_group_points_grad_ex runs (spc_group_points_grad when there is no workspace)."""
    if not workspace:
        return "atomic"
    if C < K["EX_MIN_C"]:
        return "atomic, ex fallback C<4"
    if N <= K["GB_MAX_N"] and N > K["EX_POINTS_PER_C"] * C:
        return "atomic, ex fallback N>512C"
    return "gather" if N > K["GB_MAX_N"] else "csr"


def plan_bn(K, C, S, aligned):
    """bn_relu.cu plan_bn: (vec, splits)."""
    splits = _cdiv(K["BN_CTAS_PER_SM"] * K["kNumSMs"], C)
    splits = max(1, min(splits, K["BN_MAX_SPLITS"], _cdiv(S, K["BN_THREADS"] * 4)))
    chunk = (_cdiv(S, splits) + 3) & ~3
    return S % 4 == 0 and aligned, _cdiv(S, chunk)


def plan_interp(K, B, C, m, n):
    """interp.cu spc_three_interpolate: (CT before the halving loop, CT after it; 0 = the kernel without smem)."""
    CT = min(K["TI_FWD_BYTES"] // (4 * m) if m > 0 else 0, K["TI_FWD_CT_MAX"], C)
    CT0 = CT
    xchunks = _cdiv(n, K["TI_THREADS"] * 4)
    while CT > K["TI_FWD_CT_MIN"] and xchunks * _cdiv(C, CT) * B < K["TI_FWD_WAVES"] * K["kNumSMs"]:
        CT //= 2
    return CT0, CT


# ---- data -----------------------------------------------------------------------------------------------------------
def _seed(name):
    return zlib.crc32(name.encode()) & 0x7FFFFFFF


def _gen(name, dev):
    return torch.Generator(device=dev).manual_seed(_seed(name))


def _ints(lo, hi, shape, g, dev):
    """Integers in [lo, hi] as float64."""
    return torch.randint(lo, hi + 1, shape, generator=g, device=dev, dtype=torch.int32).double()


def _k8(shape, g, dev):
    """k/8, k in [-8, 8], as fp32."""
    return (_ints(-8, 8, shape, g, dev) / 8).float()


def _is_f32(t):
    return torch.equal(t.float().double(), t)


def _poison(shape):
    """Leave a NaN-filled block in the caching allocator, so that an output allocated with torch.empty right after
    starts out as NaN: an element a kernel fails to write cannot pass by holding an earlier result."""
    torch.full(shape, float("nan"), device=DEV)


def _expect_equal(got, want, what):
    got, want = got.double(), want.double()
    bad = got != want
    if not bool(bad.any()):
        return
    i = int(bad.flatten().nonzero()[0])
    raise AssertionError("%s: %d of %d differ, first at flat index %d: %r != %r" % (
        what, int(bad.sum()), bad.numel(), i, float(got.flatten()[i]), float(want.flatten()[i])))


# ---- group_points / group_points_grad -------------------------------------------------------------------------------
# (id, B, C, N, npoint, nsample, hubs): the ball-query padding repeats the first hit of a row, here `first % hubs`,
# so a few low point indices collect long position lists.  Comments: forward / atomic / list-based plan.
GROUP_CASES = [
    ("csr-ct4-h1", 3, 7, 512, 256, 16, 10),            # staged vec4 / one chunk / CT=4, lists in smem, C%4 != 0
    ("csr-ct3", 2, 7, 1000, 320, 16, 8),               # S=5120: Sp in 4097..5461 -> CT=3, channel tiles 3+3+1
    ("csr-ct2-nobulk", 2, 5, 1000, 455, 18, 6),        # S=8190: staged scalar / CT=2 without bulk copy
    ("csr-ct1-h1", 1, 5, 333, 1024, 16, 5),            # ct*N % 4 != 0: staging without bulk copy / 4 chunks / CT=1
    ("csr-h2-nobulk", 2, 6, 1000, 1001, 27, 12),       # S=27027: H=2 without bulk copy, ragged
    ("csr-h2-global", 2, 8, 4096, 1024, 32, 40),       # S=32768: H=2, lists in global memory
    ("csr-h3-ragged-smem", 1, 8, 2000, 1537, 32, 30),  # S=49184: H=3 (16400, 16400, 16384), lists in smem
    ("csr-ct2-global-n8192", 1, 16, 8192, 512, 16, 20),  # N=8192 exactly: CT=2 with lists in global memory
    ("csr-ct4-n8192", 2, 16, 8192, 256, 16, 20),       # N=8192: CT=4, lists in smem
    ("ex-fallback-n3000-c5", 2, 5, 3000, 100, 16, 10),  # N > 512*C: _ex takes the atomic kernel
    ("gather-n8193-1tile", 2, 8, 8193, 256, 32, 30),   # N=8193: point-owned gather, one 8-channel tile
    ("gather-ragged-tile", 1, 13, 9000, 300, 64, 3),   # tiles 8+5, hubs with lists of hundreds
    ("gather-16tiles", 1, 128, 8193, 64, 16, 4),
    ("unstaged-vec4", 2, 3, 60000, 1024, 16, 50),      # N > 51200: unstaged forward / unstaged atomic, C<4 fallback
    ("unstaged-scalar", 1, 4, 51201, 37, 7, 5),        # S=259
    # config 5 (tools/bench_train.py: 4 scenes, SA npoint x2, x4, x5), once each
    ("c5-80k-sa1-xyz", 4, 3, 80000, 4096, 64, 64),
    ("c5-80k-sa1-feat", 4, 1, 80000, 4096, 64, 64),
    ("c5-80k-sa2", 4, 128, 4096, 2048, 32, 64),        # H=3, lists in global memory
    ("c5-160k-sa2", 4, 128, 8192, 4096, 32, 64),       # H=6
    ("c5-160k-sa3", 4, 256, 4096, 2048, 16, 64),       # H=2, lists in global memory
    ("c5-200k-sa1-xyz", 4, 3, 200000, 10240, 64, 64),
    ("c5-200k-sa1-feat", 4, 1, 200000, 10240, 64, 64),
    ("c5-200k-sa2", 4, 128, 10240, 5120, 32, 64),      # N > 8192: gather with 16 channel tiles
]


def make_group_idx(case):
    """Ball-query-like (B, npoint, nsample) table: a random prefix of hits, the rest the padding point; a third of the
    rows full; the last point and point 0 referenced."""
    name, B, C, N, npoint, ns, hubs = case
    rng = np.random.default_rng(_seed(name))
    idx = rng.integers(0, N, (B, npoint, ns))
    cnt = rng.integers(1, ns + 1, (B, npoint, 1))
    cnt[:, ::3] = ns
    pad = idx[:, :, :1] % hubs
    idx = np.where(np.arange(ns) < cnt, idx, pad)
    idx[:, 0, 0] = N - 1
    idx[:, -1, -1] = 0
    return idx.astype(np.int32)


def group_branches(K, case, idx):
    name, B, C, N, npoint, ns, hubs = case
    S = npoint * ns
    br = set()
    staged, CT, nchunks = plan_group(K, B, C, N, S)
    kind = "vec4" if S % 4 == 0 else "scalar"
    if staged:
        bulk = all(((b * C + c0) * N) % 4 == 0 and (min(CT, C - c0) * N) % 4 == 0
                   for b in range(B) for c0 in range(0, C, CT))
        br.add("fwd staged " + kind if bulk else "fwd staged, no bulk copy")
    else:
        br.add("fwd unstaged " + kind)
    routes = {grad_route(K, C, N, False), grad_route(K, C, N, True),
              grad_route(K, C, N, C >= K["EX_MIN_C"])}          # spc_group_points_grad, _ex, and _ext's choice
    for r in routes:
        if r.startswith("atomic"):
            br.add(r.replace("atomic, ", ""))
            if not staged:
                br.add("atomic unstaged")
            else:
                br.add("atomic staged, one chunk" if nchunks == 1 else "atomic staged, several chunks")
        elif r == "gather":
            tiles = _cdiv(C, K["GL_CT"])
            br.add("gather %d tile%s" % (tiles, "s" if tiles > 1 else ""))
            if C % K["GL_CT"]:
                br.add("gather ragged tile")
            if max(np.bincount(idx[b].ravel(), minlength=N).max() for b in range(B)) > K["GL_LONG"]:
                br.add("gather long lists")
            if N == K["GB_MAX_N"] + 1:
                br.add("gather N=8193")
        else:
            H, Sp, GCT, smem = plan_group_grad(K, C, N, S)
            bulk = S % 8 == 0
            hs = "H=%d" % H if H < 3 else "H>=3"
            br |= {"csr CT=%d" % GCT, "csr " + hs,
                   "csr<%d,%s>" % (GCT, "smem" if smem else "global"),
                   "csr lists " + ("smem" if smem else "global"), "csr bulk" if bulk else "csr no bulk"}
            if S % Sp:
                br.add("csr ragged last partition, " + hs)
            if not bulk and H >= 2:
                br.add("csr no bulk, H>=2")
            if N == K["GB_MAX_N"]:
                br.add("csr N=8192")
            flat = idx.reshape(B, S)
            if max(np.bincount(flat[b, h * Sp:(h + 1) * Sp], minlength=N).max()
                   for b in range(B) for h in range(H)) > K["GG_SHORT"]:
                br.add("csr long lists")
    if name.startswith("c5-"):
        br.add(name)
    return br


@pytest.mark.gpu
@pytest.mark.parametrize("case", GROUP_CASES, ids=[c[0] for c in GROUP_CASES])
def test_group_points_exact(case):
    """group_points == the gather, and group_points_grad == the float64 scatter_add_, bit for bit, through _ext and
    through both library entry points on the same data: spc_group_points_grad (atomic kernels) and
    spc_group_points_grad_ex with a workspace (list-based kernels, or its fallbacks)."""
    from spacap3d_b200 import _ext, _lib
    name, B, C, N, npoint, ns, hubs = case
    S = npoint * ns
    assert S * 8 < FP32_UNITS
    idx = torch.from_numpy(make_group_idx(case)).to(DEV)
    g = _gen(name, DEV)
    points = _k8((B, C, N), g, DEV)
    li = idx.view(B, 1, S).long().expand(B, C, S)
    _poison((B, C, S))
    out = _ext.group_points(points, idx)
    _expect_equal(out.view(B, C, S), torch.gather(points, 2, li), "group_points")
    del out
    go = _k8((B, C, npoint, ns), g, DEV)
    want = torch.zeros(B, C, N, dtype=torch.float64, device=DEV).scatter_add_(2, li, go.view(B, C, S).double())
    _poison((B, C, N))
    _expect_equal(_ext.group_points_grad(go, idx, N), want, "_ext.group_points_grad")
    stream = torch.cuda.current_stream().cuda_stream
    got = torch.full((B, C, N), float("nan"), device=DEV)
    _lib.call("spc_group_points_grad", go.data_ptr(), idx.data_ptr(), B, C, N, npoint, ns, got.data_ptr(), stream)
    _expect_equal(got, want, "spc_group_points_grad")
    nbytes = _lib.load().spc_group_points_grad_workspace_bytes(B, N, npoint, ns)
    assert nbytes > 0
    ws = torch.empty((nbytes + 3) // 4, dtype=torch.int32, device=DEV)
    got.fill_(float("nan"))
    _lib.call("spc_group_points_grad_ex", go.data_ptr(), idx.data_ptr(), B, C, N, npoint, ns, got.data_ptr(),
              ws.data_ptr(), nbytes, stream)
    _expect_equal(got, want, "spc_group_points_grad_ex")


# ---- gather_points_grad ---------------------------------------------------------------------------------------------
GATHER_CASES = [                  # (id, B, C, N, M)
    ("c70-m1000", 2, 70, 500, 1000),      # C > 64: the channel-stride loop; M % 256 != 0
    ("c130-dups", 1, 130, 50, 3000),      # every point ~60 times
    ("c3-m256", 3, 3, 1000, 256),
]


def make_gather_idx(case):
    name, B, C, N, M = case
    rng = np.random.default_rng(_seed(name))
    idx = rng.integers(0, N, (B, M))
    idx[:, ::2] = rng.integers(0, 4, (B, (M + 1) // 2))     # heavy duplicates on four points
    idx[:, -1] = N - 1
    return idx.astype(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("case", GATHER_CASES, ids=[c[0] for c in GATHER_CASES])
def test_gather_points_grad_exact(case):
    from spacap3d_b200 import _ext
    name, B, C, N, M = case
    idx = torch.from_numpy(make_gather_idx(case)).to(DEV)
    go = _k8((B, C, M), _gen(name, DEV), DEV)
    want = torch.zeros(B, C, N, dtype=torch.float64, device=DEV).scatter_add_(
        2, idx.view(B, 1, M).long().expand(B, C, M), go.double())
    _poison((B, C, N))
    _expect_equal(_ext.gather_points_grad(go, idx, N), want, "gather_points_grad")


# ---- three_interpolate / three_interpolate_grad ---------------------------------------------------------------------
INTERP_CASES = [                  # (id, B, C, m, n)
    ("ct-halving-grad-smem", 1, 64, 256, 999),       # CT 32 -> 4; n % 4 != 0; grad rows 8 KB
    ("grad-smem-40k", 1, 8, 1280, 300),              # grad rows exactly 40 KB: no opt-in
    ("staged-nobulk-grad-optin", 2, 21, 2001, 1500),  # last channel tile of one odd row: no bulk copy; 64 KB opt-in
    ("grad-optin-96k", 1, 9, 3072, 2048),            # exactly 96 KB
    ("grad-global-c70", 2, 70, 3073, 500),           # global atomics, C > 64 (channel-stride loop)
    ("nosmem-grad-global", 2, 10, 20000, 777),       # m > 16384: forward without smem
    ("n0-smem", 2, 5, 100, 0),                       # n = 0: the gradient must be zeros, on both sides of 96 KB
    ("n0-global", 2, 5, 4000, 0),
    ("c5-200k-fp2", 4, 256, 2560, 5120),             # FP2 at 200k points: 80 KB opt-in
]


def make_interp_idx_w(case):
    name, B, C, m, n = case
    rng = np.random.default_rng(_seed(name))
    idx = rng.integers(0, m, (B, n, 3))
    idx[:, ::7, 1] = idx[:, ::7, 0]                      # repeated neighbours
    idx[:, ::11, :] = idx[:, ::11, :1]                   # one neighbour three times
    w = rng.integers(0, 17, (B, n, 3)) / 16.0            # rows do not sum to 1
    w[:, ::5, 2] = 0.0
    w[:, ::13, :] = 0.0
    if n:
        idx[:, 0] = (m - 1, 0, m - 1)
        w[:, 1] = (0.5, 0.25, 0.25)                      # some rows do sum to 1
    return idx.astype(np.int32), w.astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("case", INTERP_CASES, ids=[c[0] for c in INTERP_CASES])
def test_three_interpolate_exact(case):
    from spacap3d_b200 import _ext
    name, B, C, m, n = case
    assert 3 * n * 2 ** 7 < FP32_UNITS
    idx_np, w_np = make_interp_idx_w(case)
    idx, w = torch.from_numpy(idx_np).to(DEV), torch.from_numpy(w_np).to(DEV)
    g = _gen(name, DEV)
    points, go = _k8((B, C, m), g, DEV), _k8((B, C, n), g, DEV)
    li = idx.view(B, 1, 3 * n).long().expand(B, C, 3 * n)
    if n:
        want = (torch.gather(points.double(), 2, li).view(B, C, n, 3) * w.double()[:, None]).sum(-1)
        _poison((B, C, n))
        _expect_equal(_ext.three_interpolate(points, idx, w), want, "three_interpolate")
    want = torch.zeros(B, C, m, dtype=torch.float64, device=DEV).scatter_add_(
        2, li, (go.double()[..., None] * w.double()[:, None]).reshape(B, C, 3 * n))
    _poison((B, C, m))
    _expect_equal(_ext.three_interpolate_grad(go, idx, w, m), want, "three_interpolate_grad")


# ---- BatchNorm + ReLU (+ max-pool), training mode -------------------------------------------------------------------
BN_CASES = [                      # shape (B, C, ...): the statistics run over every dimension but 1
    dict(id="vec-1split", shape=(2, 8, 512)),
    dict(id="vec-splits", shape=(2, 16, 8192)),
    dict(id="vec-splits-eps3a2", shape=(4, 8, 2048), eps3=True),
    dict(id="scalar-splits-offset4", shape=(2, 8, 4096), offset=True),    # y 4 bytes past 16-byte alignment
    dict(id="scalar-S2047", shape=(16, 5, 2047)),
    dict(id="C1-64splits", shape=(4, 1, 65536)),
    dict(id="BC65535", shape=(3, 21845, 16)),
    dict(id="BC80000-slices", shape=(2, 40000, 16)),                     # two apply launches of one batch row
    dict(id="c5-160k-bn", shape=(4, 64, 8192, 64), dz1=True),            # M = 2^21
]
POOL_CASES = [                    # shape (B, C, npoint, nsample)
    dict(id="ns16-below-cta", shape=(2, 6, 100, 16)),
    dict(id="ns32-below-cta", shape=(3, 5, 64, 32)),
    dict(id="ns64-below-cta", shape=(2, 4, 48, 64)),
    dict(id="ns16-ctas", shape=(2, 8, 1024, 16)),
    dict(id="ns32-ctas-np1000", shape=(2, 6, 1000, 32)),
    dict(id="ns64-ctas-eps3a2", shape=(4, 4, 512, 64), eps3=True),
    dict(id="ns16-BC66000-slices", shape=(2, 33000, 2, 16)),             # two pool launches of one batch row
    dict(id="c5-200k-bnpool", shape=(4, 128, 10240, 64), dz1=True),       # M = 2 621 440
]
BN_MOMENTUM = 0.125
SMALL = 2 ** 22                   # cases up to this many elements are drawn on the CPU (and checked there)
_BLOCK = (-2.0, 2.0, -1.0, -1.0, -1.0, -1.0, 1.0, 1.0, 1.0, 1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0)


def _bn_dev(c):
    return "cpu" if math.prod(c["shape"]) <= SMALL else DEV


def make_bn(c, dev, pool=False):
    """Exact operands of one BatchNorm case (float64 tensors on `dev`; y also as fp32)."""
    shape = c["shape"]
    B, C = shape[:2]
    S = math.prod(shape[2:])
    M = B * S
    assert M % len(_BLOCK) == 0
    g = _gen(c["id"], dev)
    t = torch.tensor(_BLOCK, dtype=torch.float32, device=dev)[
        torch.argsort(torch.rand(C, M, generator=g, device=dev), dim=1) % len(_BLOCK)]
    first0 = (t == 0).to(torch.uint8).argmax(1)                    # move a zero to (b=0, s=0): the kernel's shift
    rows = torch.arange(C, device=dev)
    t[rows, first0] = t[:, 0].clone()
    t[:, 0] = 0
    e = torch.full((C,), -1.0, device=dev, dtype=torch.float64) if c.get("eps3") else _ints(-3, 2, (C,), g, dev)
    a = 2.0 ** e
    mu = _ints(-64, 64, (C,), g, dev) / 16
    y = (mu[:, None] + a[:, None] * t.double()).view(C, B, S).transpose(0, 1).contiguous().view(shape)
    del t
    eps = 3 * 2.0 ** -2 if c.get("eps3") else 0.0                 # 3 a^2: var + eps = (2a)^2, xhat = t / 2
    s = 0.5 if c.get("eps3") else 1.0
    sign = torch.where(torch.arange(C, device=dev) % 2 == 1, -1.0, 1.0).double()    # negative gamma on odd channels
    gamma = sign * 2.0 ** _ints(-1, 1, (C,), g, dev)
    t0 = _ints(-2, 2, (C,), g, dev)
    t0[0] = 0                                                        # beta = 0
    allneg = sign * _ints(2, 3, (C,), g, dev)                        # z = gamma s (t - t0) <= 0 for every t
    mode = torch.arange(C, device=dev) % 3
    beta = torch.where(mode == 0, -gamma * s * t0,
                       torch.where(mode == 1, _ints(-8, 8, (C,), g, dev) / 8, -gamma * s * allneg))
    dshape = shape[:3] if pool else shape
    dz = _ints(-1, 1, dshape, g, dev) if c.get("dz1") else _ints(-2, 2, dshape, g, dev) / 2
    return dict(y=y, gamma=gamma, beta=beta, eps=eps, dz=dz, rm=_ints(-16, 16, (C,), g, dev) / 16,
                rv=_ints(1, 32, (C,), g, dev) / 16, M=M, s=s)


def _gamma_n(n):
    u = 2.0 ** -24
    return n * u / (1 - n * u)


def _bn_reference(d, pool=False):
    """Textbook two-pass BatchNorm + ReLU (+ max over the last dimension) in float64, with the exactness conditions
    asserted on the data.  Not ATen's float64 batch_norm: its Welford update divides by non-power-of-two counts and
    can leave residuals around 1e-17 that survive the cast to fp32 and flip the mask at the exact zeros."""
    y, gamma, beta, eps, dz, M = d["y"], d["gamma"], d["beta"], d["eps"], d["dz"], d["M"]
    red = tuple(i for i in range(y.dim()) if i != 1)
    bc = lambda v: v.view((1, -1) + (1,) * (y.dim() - 2))          # noqa: E731
    assert _is_f32(y) and _is_f32(gamma) and _is_f32(beta) and _is_f32(dz)
    mean = y.sum(red) / M
    var = ((y - bc(mean)) ** 2).sum(red) / M
    invstd = 1 / torch.sqrt(var + eps)
    xh = (y - bc(mean)) * bc(invstd)
    zp = bc(gamma) * xh + bc(beta)
    r = dict(mean=mean, invstd=invstd, rm=(1 - BN_MOMENTUM) * d["rm"] + BN_MOMENTUM * mean,
             rv=(1 - BN_MOMENTUM) * d["rv"] + BN_MOMENTUM * var * M / (M - 1))
    for k in ("mean", "invstd", "rm"):
        assert _is_f32(r[k]), k
    assert _is_f32(xh) and _is_f32(zp)
    stats = dict(zero=bool((zp == 0).any()))
    if pool:
        am = zp.argmax(-1, keepdim=True)                              # ties: the first maximal slot (documented)
        zmax = zp.gather(-1, am)
        stats.update(ties=bool(((zp == zmax).sum(-1) > 1).any()), nonpos=bool((zmax <= 0).any()),
                     pos=bool((zmax > 0).any()))
        r.update(pooled=zmax.clamp_min(0).squeeze(-1), argmax=am.squeeze(-1), ymax=y.gather(-1, am).squeeze(-1))
        dm = torch.zeros_like(y).scatter_(-1, am, torch.where(zmax > 0, dz[..., None], 0.0))
        del zmax, am
    else:
        r["z"] = zp.clamp_min(0)
        dm = torch.where(zp > 0, dz, 0.0)
    del zp
    dbeta, dgamma = dm.sum(red), (dm * xh).sum(red)
    assert _is_f32(dbeta) and _is_f32(dgamma)
    k0, k1, gs = dbeta / M, dgamma / M, gamma * invstd
    assert _is_f32(gs)
    dy = bc(gs) * ((dm - bc(k0)) - xh * bc(k1))
    r.update(dbeta=dbeta, dgamma=dgamma, dy=dy, exact_dy=(M & (M - 1)) == 0, stats=stats)
    if r["exact_dy"]:
        # inv_M is exact: so is every step of gs * ((dm - k0) - xh * k1) if each is an fp32 value
        for name, v in (("k0", k0), ("k1", k1), ("dm - k0", dm - bc(k0)), ("xh * k1", xh * bc(k1)), ("dy", dy)):
            assert _is_f32(v), "dy intermediate %s is not an fp32 value" % name
    else:
        # The kernel evaluates inv_M = fl(1/M) (through float64: within u + 2^-53 of 1/M), k0 = fl(dbeta * inv_M),
        # k1 = fl(dgamma * inv_M), A = fl(dm - k0), B = fl(A - fl(xh * k1)) (or one fma) and dy = fl(gs * B), each
        # correctly rounded with |relative error| <= u = 2^-24; gs, xh, dm, dbeta and dgamma are exact.  The dm term
        # passes through 3 roundings, the k0 and xh*k1 terms through 5 each, so
        #     |dy - dy*| <= gamma_5 |gs| (|dm| + |k0*| + |xh k1*|),   gamma_n = n u / (1 - n u).
        # gamma_6 is used: the sixth u covers the double rounding of 1/M and this float64 reference's own rounding,
        # both below 2^-50 relative.
        r["dy_err"] = _gamma_n(6) * bc(gs.abs()) * (dm.abs() + bc(k0.abs()) + xh.abs() * bc(k1.abs()))
    return r


def _bn_analytic(c, pool=False):
    """The exactness conditions of a case from its generator parameters alone: every partial sum of the statistics
    and of the backward reduction below 2^24 units of its grid, and, when M is a power of two, every intermediate of
    dy on the grid 2^-(q_dz + 2 q_x) / M with magnitude below 2^24 such units."""
    shape = c["shape"]
    M = shape[0] * math.prod(shape[2:])
    assert M % len(_BLOCK) == 0 and M < 2 ** 22
    assert 2 * M < FP32_UNITS and 4 * M < FP32_UNITS                # sum |y-K| <= 2Ma, sum (y-K)^2 <= 4Ma^2
    q_dz, dz_max = (0, 1.0) if c.get("dz1") else (1, 1.0)
    q_x, x_max = (1, 1.0) if c.get("eps3") else (0, 2.0)            # xhat = s * t
    assert M * dz_max * 2 ** q_dz < FP32_UNITS                       # dbeta
    assert M * dz_max * x_max * 2 ** (q_dz + q_x) < FP32_UNITS       # dgamma
    if M & (M - 1) == 0:
        # |k0| <= dz_max, |k1| <= dz_max x_max, |(dm - k0) - xh k1| <= dz_max (2 + x_max^2); gs = gamma / a is a power
        # of two, so dy = gs * (...) is exact when (...) is
        assert dz_max * (2 + x_max ** 2) * 2 ** (q_dz + 2 * q_x) * M < FP32_UNITS
        return True
    return False


def _to_dev32(d, offset=False):
    y32 = d["y"].float().to(DEV)
    assert y32.is_contiguous()
    if offset:
        store = torch.empty(y32.numel() + 1, device=DEV)
        store[1:] = y32.flatten()
        y32 = store[1:].view(y32.shape)
        assert y32.data_ptr() % 16 == 4 and y32.is_contiguous()
    f = lambda k: d[k].float().to(DEV)                              # noqa: E731
    return y32, f("gamma"), f("beta"), f("rm"), f("rv"), f("dz")


def _check_bn_outputs(ref, got, what):
    for k, v in got.items():
        if k == "rv":
            want = ref["rv"].to(DEV)
            ulp = 2.0 ** (torch.floor(torch.log2(want.abs())) - 23)
            assert bool(((v.double() - want).abs() <= ulp).all()), (what, "running_var", v, want)
        elif k == "dy" and not ref["exact_dy"]:
            err = (v.double() - ref["dy"].to(DEV)).abs()
            bound = ref["dy_err"].to(DEV)
            assert bool((err <= bound).all()), (what, "dy", float((err - bound).max()))
        else:
            _expect_equal(v, ref[k].to(DEV), "%s %s" % (what, k))


@pytest.mark.gpu
@pytest.mark.parametrize("c", BN_CASES, ids=[c["id"] for c in BN_CASES])
def test_bn_relu_train_exact(c):
    """bn_relu_train_forward / _backward: z, save_mean, save_invstd, running_mean, dgamma, dbeta bit for bit,
    running_var within one ulp, dy bit for bit (M a power of two) or within its derived bound."""
    from spacap3d_b200 import _ext
    d = make_bn(c, _bn_dev(c))
    ref = _bn_reference(d)
    y, gamma, beta, rm, rv, dz = _to_dev32(d, c.get("offset", False))
    _poison(y.shape)
    z, mean, invstd = _ext.bn_relu_train_forward(y, gamma, beta, rm, rv, BN_MOMENTUM, d["eps"])
    _poison(y.shape)
    dy, dgamma, dbeta = _ext.bn_relu_train_backward(dz, y, gamma, beta, mean, invstd)
    _check_bn_outputs(ref, dict(z=z, mean=mean, invstd=invstd, rm=rm, rv=rv, dy=dy, dgamma=dgamma, dbeta=dbeta),
                      c["id"])


@pytest.mark.gpu
@pytest.mark.parametrize("c", POOL_CASES, ids=[c["id"] for c in POOL_CASES])
def test_bn_relu_maxpool_exact(c):
    """bn_relu_maxpool_train_forward / _backward: pooled, the winning slot (the first on ties), the pre-BN value
    there, the statistics and running buffers, dy, dgamma and dbeta against the float64 evaluation."""
    from spacap3d_b200 import _ext
    d = make_bn(c, _bn_dev(c), pool=True)
    ref = _bn_reference(d, pool=True)
    y, gamma, beta, rm, rv, dpool = _to_dev32(d)
    pooled, argmax, ymax, mean, invstd = _ext.bn_relu_maxpool_train_forward(y, gamma, beta, rm, rv, BN_MOMENTUM,
                                                                            d["eps"])
    _poison(y.shape)
    dy, dgamma, dbeta = _ext.bn_relu_maxpool_train_backward(dpool, argmax, ymax, y, gamma, beta, mean, invstd)
    _check_bn_outputs(ref, dict(pooled=pooled, argmax=argmax, ymax=ymax, mean=mean, invstd=invstd, rm=rm, rv=rv,
                                dy=dy, dgamma=dgamma, dbeta=dbeta), c["id"])


@pytest.mark.gpu
def test_bn_relu_maxpool_misaligned_y_unsupported():
    """The pooled kernels read y with 16-byte loads: a y that is not 16-byte aligned is refused, nothing launched."""
    from spacap3d_b200 import _ext, _lib
    B, C, npoint, ns = 2, 4, 64, 16
    store = torch.zeros(B * C * npoint * ns + 1, device=DEV)
    y = store[1:].view(B, C, npoint, ns)
    gamma, beta = torch.ones(C, device=DEV), torch.zeros(C, device=DEV)
    with pytest.raises(_lib.SpcUnsupported):
        _ext.bn_relu_maxpool_train_forward(y, gamma, beta, None, None, BN_MOMENTUM, 1e-5)
    dpool = torch.zeros(B, C, npoint, device=DEV)
    argmax = torch.zeros(B, C, npoint, dtype=torch.uint8, device=DEV)
    mean, invstd = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    with pytest.raises(_lib.SpcUnsupported):
        _ext.bn_relu_maxpool_train_backward(dpool, argmax, dpool, y, gamma, beta, mean, invstd)


def bn_branches(K, c, pool=False):
    shape = c["shape"]
    B, C = shape[:2]
    S = math.prod(shape[2:])
    br = set()
    if pool:
        ns, npoint = shape[3], shape[2]
        cover = (K["BN_THREADS"] // 32) * (32 // (ns // 4)) * K["BP_UNR"]
        br |= {"pool ns=%d" % ns, "pool below one CTA" if npoint < cover else "pool several CTAs"}
        if npoint & (npoint - 1):
            br.add("pool npoint not a power of two")
    else:
        vec, splits = plan_bn(K, C, S, not c.get("offset", False))
        br.add("bn %s, %s" % ("vector" if vec else "scalar", "one split" if splits == 1 else "several splits"))
        if S % 4:
            br.add("bn S%4!=0")
        if C == 1 and splits == K["BN_MAX_SPLITS"]:
            br.add("bn C=1, 64 splits")
        if B * C == 65535:
            br.add("bn B*C=65535")
    if B > max(1, K["BN_SLICE_ROWS"] // C):
        br.add("sliced apply")
    if c.get("eps3"):
        br.add("bn eps=3a^2")
    if c["id"].startswith("c5-"):
        br.add(c["id"])
    return br


def interp_branches(K, case):
    name, B, C, m, n = case
    br = set()
    if n:
        CT0, CT = plan_interp(K, B, C, m, n)
        br.add("interp fwd no smem" if CT == 0 else "interp fwd staged")
        if 0 < CT < CT0:
            br.add("interp fwd CT halved")
    smem = K["TI_CT"] * m * 4
    kind = ("smem" if smem <= K["TI_GRAD_OPTIN"] else "opt-in smem") if smem <= K["TI_GRAD_SMEM_MAX"] else "global"
    br.add("interp grad %s%s" % (kind, ", n=0" if n == 0 else ""))
    if name.startswith("c5-"):
        br.add(name)
    return br


# Every branch named in the plan functions that the training path can reach, and the config-5 shapes.
BRANCHES = {
    "fwd staged vec4", "fwd staged scalar", "fwd staged, no bulk copy", "fwd unstaged vec4", "fwd unstaged scalar",
    "atomic staged, one chunk", "atomic staged, several chunks", "atomic unstaged",
    "ex fallback C<4", "ex fallback N>512C",
    "csr CT=1", "csr CT=2", "csr CT=3", "csr CT=4", "csr H=1", "csr H=2", "csr H>=3",
    "csr ragged last partition, H=2", "csr ragged last partition, H>=3",
    # the instantiations the plan can pick: lists of CT=3, 4 (Sp <= 5456) always fit in shared memory
    "csr<1,smem>", "csr<2,smem>", "csr<3,smem>", "csr<4,smem>", "csr<1,global>", "csr<2,global>",
    "csr lists smem", "csr lists global", "csr bulk", "csr no bulk", "csr no bulk, H>=2", "csr long lists",
    "csr N=8192",
    "gather 1 tile", "gather 16 tiles", "gather ragged tile", "gather long lists", "gather N=8193",
    "gpg C>64", "gpg duplicates", "gpg M%256!=0",
    "interp fwd CT halved", "interp fwd staged", "interp fwd no smem",
    "interp grad smem", "interp grad opt-in smem", "interp grad global", "interp grad smem, n=0",
    "interp grad global, n=0",
    "bn vector, one split", "bn vector, several splits", "bn scalar, several splits", "bn S%4!=0",
    "bn C=1, 64 splits", "bn B*C=65535", "bn eps=3a^2", "sliced apply",
    "pool ns=16", "pool ns=32", "pool ns=64", "pool below one CTA", "pool several CTAs",
    "pool npoint not a power of two",
    "c5-80k-sa1-xyz", "c5-80k-sa1-feat", "c5-80k-sa2", "c5-160k-sa2", "c5-160k-sa3", "c5-160k-bn",
    "c5-200k-sa1-xyz", "c5-200k-sa1-feat", "c5-200k-sa2", "c5-200k-fp2", "c5-200k-bnpool",
}


# =================================================================================================================
def test_generators_meet_preconditions():
    """Every case of this file, in float64 on the CPU: the scatter and interpolation bounds from the shapes, the data
    features the cases claim (duplicates, zero weights, rows not summing to 1), and every exactness condition of the
    BatchNorm cases -- on the drawn data for the small ones, analytically for the large ones -- including each
    intermediate of dy being an fp32 value, exact zeros of z, negative gamma, beta = 0, ties and non-positive groups."""
    for case in GROUP_CASES:
        assert case[4] * case[5] * 8 < FP32_UNITS, case[0]                 # S terms of k/8 at most per output
        idx = make_group_idx(case)
        assert idx.min() >= 0 and idx.max() < case[3]
    for case in GATHER_CASES:
        name, B, C, N, M = case
        assert M * 8 < FP32_UNITS
        idx = make_gather_idx(case)
        assert idx.min() >= 0 and idx.max() < N
        assert all(np.bincount(idx[b]).max() > 1 for b in range(B))
    for case in INTERP_CASES:
        name, B, C, m, n = case
        assert 3 * 2 ** 7 < FP32_UNITS and 3 * n * 2 ** 7 < FP32_UNITS
        idx, w = make_interp_idx_w(case)
        if n:
            assert idx.min() >= 0 and idx.max() < m
            assert ((w * 16) == np.round(w * 16)).all() and w.min() >= 0 and w.max() <= 1
            assert (w == 0).any() and (idx[..., 0] == idx[..., 1]).any()
            assert (w.sum(-1) != 1).any() and (w.sum(-1) == 1).any()
    seen = {}
    for pool, cases in ((False, BN_CASES), (True, POOL_CASES)):
        for c in cases:
            exact = _bn_analytic(c, pool)
            if _bn_dev(c) != "cpu":
                continue
            d = make_bn(c, "cpu", pool)
            r = _bn_reference(d, pool)          # asserts every intermediate on the drawn data
            assert r["exact_dy"] == exact
            K0 = d["y"].flatten(2)[0, :, 0]                 # y at (b=0, s=0): the kernel's shift is the mean
            assert torch.equal(r["mean"], K0), c["id"]
            bc = lambda v: v.view((1, -1) + (1,) * (d["y"].dim() - 2))          # noqa: E731
            t = (d["y"] - bc(K0)) * bc(r["invstd"]) / d["s"]
            assert torch.equal(t, t.round()) and float(t.abs().max()) == 2, c["id"]
            st = r["stats"]
            assert st["zero"], c["id"]
            assert bool((d["gamma"] < 0).any()) or d["gamma"].numel() == 1, c["id"]
            assert bool((d["beta"] == 0).any()), c["id"]
            if pool:
                assert st["ties"] and st["nonpos"] and st["pos"], (c["id"], st)
            seen[c["id"]] = exact
    assert True in seen.values() and False in seen.values()   # both the exact and the bounded dy are exercised


def test_cases_reach_their_branches():
    """With the launch plans restated from csrc/group.cu, interp.cu and bn_relu.cu (constants read from the sources),
    every branch in BRANCHES is taken by at least one case, and the config-5 shapes take the branches they are here
    for."""
    K = _constants()
    reached = {}
    for case in GROUP_CASES:
        reached[case[0]] = group_branches(K, case, make_group_idx(case))
    for name, B, C, N, M in GATHER_CASES:
        br = set()
        if C > 64:
            br.add("gpg C>64")
        if M % 256:
            br.add("gpg M%256!=0")
        if M > N:
            br.add("gpg duplicates")
        reached["gpg " + name] = br
    for case in INTERP_CASES:
        reached["interp " + case[0]] = interp_branches(K, case)
    for c in BN_CASES:
        reached["bn " + c["id"]] = bn_branches(K, c)
    for c in POOL_CASES:
        reached["pool " + c["id"]] = bn_branches(K, c, pool=True)
    union = set().union(*reached.values())
    assert not BRANCHES - union, sorted(BRANCHES - union)
    # what the config-5 shapes are here for
    assert {"csr H>=3", "csr ragged last partition, H>=3", "csr<1,global>"} <= reached["c5-80k-sa2"]
    assert plan_group_grad(K, 128, 8192, 4096 * 32)[0] == 6
    assert "csr ragged last partition, H>=3" in reached["c5-160k-sa2"]
    assert {"csr H=2", "csr<1,global>"} <= reached["c5-160k-sa3"]
    for n in ("c5-80k-sa1-xyz", "c5-80k-sa1-feat", "c5-200k-sa1-xyz", "c5-200k-sa1-feat"):
        assert {"fwd unstaged vec4", "atomic unstaged"} <= reached[n]
    assert {"gather 16 tiles", "gather long lists"} <= reached["c5-200k-sa2"]
    assert "interp grad opt-in smem" in reached["interp c5-200k-fp2"]
    assert "pool several CTAs" in reached["pool c5-200k-bnpool"]
    assert "sliced apply" in reached["bn BC80000-slices"] and "sliced apply" in reached["pool ns16-BC66000-slices"]
    assert "sliced apply" not in reached["bn BC65535"]
    assert plan_bn(K, 64, 8192 * 64, True) == (True, 10)
