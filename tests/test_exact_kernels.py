"""The tensor-core kernels bit for bit, on data where no rounding happens.

The fused set abstraction (csrc/sa_inline.cu, csrc/sa_fused.cu) and pm_linear (csrc/pm_linear.cu) accumulate in fp32
on the tensor cores in an unspecified order, so on random data they legitimately differ from any reference by
rounding, and test_sa_fused_gpu.py / test_pm_linear_gpu.py can only hold them to tolerances.  Here every operand lies
on a dyadic grid with so few significant bits that
  * every product is exact,
  * every partial sum is exact in fp32, in any order,
  * every value the kernels keep in 16 bits (H1, H2, G, Y_hi / Y_lo) is an fp16 value or an exact fp16 (hi, lo) pair,
so each output has exactly one correct value, the float64 evaluation, and any difference is a bug.  Two outputs are,
by definition, a rounding of such an exact fp32 value: the fused kernel's fp16 copy `out_pm` (compared with the fp16
rounding of the exact result) and the L2-normalised outputs of the voting tail (compared within a bound derived from
fp32 rounding, next to the test).

Accumulator margin.  In units of the finest grid step of its terms, the sum of the magnitudes of every dot product's
terms stays below 2^22: two bits inside fp32's 24, so an accumulator that aligns its addends to the largest one and
keeps 24 bits loses nothing.  How the sm_100a tensor core aligns and truncates while it accumulates has not been
measured; this margin is a design assumption, not a measured fact.

The fp16 (hi, lo) operand pairs (layer 0 of the in-line form, pm_linear) are covered one operand at a time: data whose
INPUTS have non-zero lo parts use fp16-exact weights, and the converse, so the product lo.lo that the kernels drop is
exactly zero.  Layer 0 of the in-line form must land on the fp16 grid although its lo parts are small, which takes
cancellation: inputs 1024 + d/4 against a bias of -1024 * sum(w) (input lo parts, bias lo part), or two feature
channels carrying the same values with weights H + l and -hi(H + l) (weight lo parts).

The CPU-only test_generators_meet_preconditions checks all of the above on every case in float64; the GPU tests compare
the kernels with the same float64 evaluation by torch.equal.
"""
import warnings

import numpy as np
import pytest
import torch

DEV = "cuda:0"
ACC_UNITS = 2 ** 22              # bound on a dot product's sum of |terms|, in units of its finest grid step


# ---- float64 helpers (CPU or GPU tensors) -----------------------------------------------------------------------
def _q(t):
    """The smallest q >= 0 such that every element of t is a multiple of 2^-q."""
    t = t.abs()
    for q in range(60):
        s = t * 2.0 ** q
        if bool((s == s.floor()).all()):
            return q
    raise AssertionError("values are not on a dyadic grid")


def _split16(t):
    """The kernels' fp16 (hi, lo) split of fp32 data (_ext.split_half, split_f16, put_group), as float64."""
    f = t.float()
    assert torch.equal(f.double(), t), "value not representable in fp32"
    hi = f.half()
    lo = (f - hi.float()).half()
    return hi.double(), lo.double()


def _is_f16(t):
    return torch.equal(t.float().half().double(), t)


def _is_f32(t):
    return torch.equal(t.float().double(), t)


class _Budget:
    """Collects the partial-sum bounds of one case: (max sum of |terms|, grid exponent of the terms)."""

    def __init__(self):
        self.sums = {}

    def add(self, name, bound, q):
        self.sums[name] = (float(bound.max()), q)

    def check(self):
        for name, (b, q) in self.sums.items():
            assert b * 2.0 ** q < ACC_UNITS, "%s: partial sums reach %g units of 2^-%d" % (name, b * 2.0 ** q, q)


# ---- fused set abstraction: all 18 compiled kernels --------------------------------------------------------------
# (C1, C2, C3, nsample, Cf, lo): lo = "x" -> the inputs carry fp16 lo parts, "w" -> the layer-0 weights do
INLINE_CASES = [
    (64, 64, 128, 64, 0, "x"), (64, 64, 128, 64, 1, "x"), (64, 64, 128, 64, 9, "x"), (64, 64, 128, 64, 13, "w"),
    (64, 64, 128, 32, 13, "x"), (64, 64, 128, 16, 9, "w"),
    (128, 128, 256, 64, 1, "x"), (128, 128, 256, 32, 9, "x"), (128, 128, 256, 16, 13, "w"),
    (128, 128, 128, 64, 13, "x"), (128, 128, 128, 32, 0, "x"), (128, 128, 128, 16, 9, "w"),
]
# (C1, C2, C3, nsample, Cf): Cf is the projection GEMM's K (a multiple of 8)
PROJ_CASES = [
    (64, 64, 128, 64, 16), (64, 64, 128, 32, 136), (64, 64, 128, 16, 24),
    (128, 128, 256, 64, 256), (128, 128, 256, 32, 128), (128, 128, 256, 16, 256),
    (128, 128, 128, 64, 64), (128, 128, 128, 32, 136), (128, 128, 128, 16, 256),
]
SA_CASES = ([("inline",) + c + (3, None) for c in INLINE_CASES] + [("proj",) + c + (None, 3, None) for c in PROJ_CASES]
            # npoint * nsample == 128: one tile per scene (the tile -> scene division path instead of tps_magic)
            + [("inline", 64, 64, 128, 16, 1, "x", 40, 8), ("proj", 128, 128, 256, 64, 24, None, 24, 2)])
SA_MIN_TILES = (0, 2, 7, 4096)   # launch hint: one tile per CTA, a few, seven, one CTA for all of them


def _sa_id(c):
    form, C1, C2, C3, ns, Cf, lo, B, npoint = c
    s = "%s-%dx%dx%d-ns%d-cf%d" % (form, C1, C2, C3, ns, Cf)
    return s + ("-%slo" % lo if lo else "") + ("-np%d-b%d" % (npoint, B) if npoint else "")


def _sparse_pm1(rng, rows, cols, nnz=8):
    """(rows, cols) with ~nnz non-zeros per row in {+-1, +-1/2} at random columns (keeps the next activation on the
    fp16 grid while every column is read by some output channel)."""
    W = np.zeros((rows, cols))
    nnz = min(nnz, cols)
    perm = rng.permutation(cols)
    for r in range(rows):                            # consecutive windows of a permutation: every column when
        c = perm[(r * nnz + np.arange(nnz)) % cols]  # rows * nnz >= cols
        W[r, c] = rng.choice([-1.0, -0.5, 0.5, 1.0], size=nnz)
    return W


def make_sa_case(form, C1, C2, C3, ns, Cf, lo, B, npoint, seed=0):
    """Exact operands of one spc_sa_fused_forward call (numpy float64, every value on its storage type's grid)."""
    rng = np.random.default_rng([seed, C1, C3, ns, Cf, B])
    npoint = npoint or 128 * 64 // ns                # 64 tiles per scene
    n = 1000
    radius = 2.0 ** int(rng.integers(-2, 2))         # power of two: (p - c) * (1 / r) is exact
    # coordinates on a grid of r/4 inside one box of side r per scene: (p - c) / r is a multiple of 1/4 in [-1, 1]
    off = rng.integers(-8, 9, size=(B, 1, 3)) * 0.5
    xyz = off + rng.integers(0, 5, size=(B, n, 3)) * (radius / 4)
    new_xyz = off + rng.integers(0, 5, size=(B, npoint, 3)) * (radius / 4)
    # ball-query-like table: a random prefix of neighbours, the rest padded with the first one
    idx = rng.integers(0, n, size=(B, npoint, ns))
    cnt = rng.integers(1, ns + 1, size=(B, npoint))
    cnt[:, ::5] = 1                                  # rows that are all one point
    idx = np.where(np.arange(ns) >= cnt[..., None], idx[..., :1], idx)
    idx[:, 1, :] = n - 1
    idx[:, min(2, npoint - 1), :3] = 0
    c = dict(form=form, C1=C1, C2=C2, C3=C3, ns=ns, Cf=Cf, B=B, n=n, npoint=npoint, radius=radius, xyz=xyz,
             new_xyz=new_xyz, idx=idx.astype(np.int32), feat=None, feat_pm=None, W0f=None)
    Wx = rng.integers(-2, 3, size=(C1, 3)).astype(np.float64)
    s = rng.integers(-8, 9, size=C1) / 4.0
    if form == "inline":
        if lo == "x":
            # features 1024 + d/4: fp16 hi plus a lo part in [-1/2, 1/2]; the bias cancels the 1024s and has a lo part
            feat = 1024 + rng.integers(-4, 5, size=(B, Cf, n)) / 4.0
            Wf = rng.integers(-1, 2, size=(C1, Cf)).astype(np.float64)
            b0 = s - 1024 * Wf.sum(1)
        else:
            # small integer features, channels 2k and 2k+1 equal; weights (H + l, -hi(H + l)), H = +-2048: only the
            # lo part l = +-1 of the first weight survives the cancellation
            feat = rng.integers(-3, 4, size=(B, Cf, n)).astype(np.float64)
            feat[:, 1::2] = feat[:, 0:Cf - Cf % 2:2]
            Wf = rng.integers(-1, 2, size=(C1, Cf)).astype(np.float64)
            npair = Cf // 2
            big = rng.choice([-1.0, 1.0], size=(C1, npair)) * (2048 + 2 * rng.integers(0, 4, size=(C1, npair)) + 1)
            Wf[:, 0:2 * npair:2] = big
            Wf[:, 1:2 * npair:2] = -big.astype(np.float32).astype(np.float16).astype(np.float64)
            b0 = s
        c.update(feat=feat if Cf else None, W0=np.concatenate([Wx, Wf], 1), b0=b0)
    else:
        c.update(feat_pm=rng.integers(-4, 5, size=(B * n, Cf)) / 2.0, W0f=_sparse_pm1(rng, C1, Cf), W0=Wx, b0=s)
    c["W1"] = _sparse_pm1(rng, C2, C1)
    c["b1"] = rng.integers(-32, 33, size=C2) / 8.0
    c["W2"] = rng.integers(-8, 9, size=(C3, C2)) / 4.0
    c["b2_offset"] = rng.integers(-64, 65, size=C3) / 32.0
    return c


def sa_reference(c, dev):
    """float64 evaluation of the fused layer: G (projected form), out (B,C3,npoint) and its fp16 copy, plus the
    checks of the preconditions.  The layer-2 bias is chosen here, from the data: minus the 30 % quantile of each
    channel's pooled maximum (plus a small offset), so that the final ReLU clips a real fraction of the outputs."""
    T = lambda a: torch.as_tensor(a, dtype=torch.float64, device=dev)       # noqa: E731
    B, n, npoint, ns, Cf = c["B"], c["n"], c["npoint"], c["ns"], c["Cf"]
    idx = torch.as_tensor(c["idx"], dtype=torch.long, device=dev)
    bi = torch.arange(B, device=dev)[:, None, None]
    xyz, new_xyz = T(c["xyz"]), T(c["new_xyz"])
    assert _is_f32(xyz) and _is_f32(new_xyz) and c["radius"] == 2.0 ** round(np.log2(c["radius"]))
    rel = (xyz[bi, idx] - new_xyz[:, :, None, :]) / c["radius"]             # (B,np,ns,3)
    assert _is_f16(rel)
    W0, b0 = T(c["W0"]), T(c["b0"])
    budget, stats = _Budget(), {}
    G = None
    if c["form"] == "inline":
        X = rel if Cf == 0 else torch.cat([rel, T(c["feat"]).transpose(1, 2)[bi, idx]], -1)
        (Xh, Xl), (Wh, Wl), (bh, bl) = _split16(X), _split16(W0), _split16(b0)
        assert float((Xl.abs() @ Wl.abs().t()).max()) == 0, "the dropped lo.lo product must be zero"
        stats.update(x_lo=bool((Xl != 0).any()), w_lo=bool((Wl != 0).any()), b_lo=bool((bl != 0).any()))
        D0 = X @ W0.t() + b0
        budget.add("layer 0", (Xh.abs() + Xl.abs()) @ Wh.abs().t() + Xh.abs() @ Wl.abs().t() + bh.abs() + bl.abs(),
                   max(_q(Xh) + _q(Wh), _q(Xl) + _q(Wh), _q(Xh) + _q(Wl), _q(bh), _q(bl)))
    else:
        Xf, W0f = T(c["feat_pm"]), T(c["W0f"])
        assert _is_f16(Xf) and _is_f16(W0f)
        G = Xf @ W0f.t()                                                     # (B*n, C1): pm_linear(PM_LINEAR)
        budget.add("projection", Xf.abs() @ W0f.abs().t(), _q(Xf) + _q(W0f))
        assert _is_f16(G), "G must be on the fp16 grid"
        Gg = G.view(B, n, -1)[bi, idx]
        D0 = Gg + rel @ W0.t() + b0                                          # the kernel's fp32 FMA chain
        budget.add("layer 0", Gg.abs() + rel.abs() @ W0.abs().t() + b0.abs(), max(_q(G), _q(rel) + _q(W0), _q(b0)))
    H1 = torch.relu(D0)
    assert _is_f16(H1), "H1 must be on the fp16 grid"
    W1, b1, W2 = T(c["W1"]), T(c["b1"]), T(c["W2"])
    assert _is_f16(W1) and _is_f16(W2) and _is_f32(b1)
    assert bool((W1 != 0).any(0).all()), "every column of W1 must be read"
    D1 = H1 @ W1.t() + b1
    budget.add("layer 1", H1 @ W1.abs().t() + b1.abs(), max(_q(H1) + _q(W1), _q(b1)))
    H2 = torch.relu(D1)
    assert _is_f16(H2), "H2 must be on the fp16 grid"
    D2 = H2 @ W2.t()
    pooled = D2.amax(2)                                                      # (B,np,C3)
    b2 = -torch.quantile(pooled.reshape(-1, pooled.shape[-1]).float(), 0.3, dim=0, interpolation="lower").double()
    b2 = b2 + T(c["b2_offset"])
    budget.add("layer 2", (H2 @ W2.abs().t()).amax(2) + b2.abs(), max(_q(H2) + _q(W2), _q(b2)))
    budget.check()
    out = torch.relu(pooled + b2).permute(0, 2, 1).contiguous()              # (B,C3,np)
    assert _is_f32(out) and _is_f32(b2)
    stats.update(relu0=float((D0 <= 0).double().mean()), relu1=float((D1 <= 0).double().mean()),
                 relu2=float((out == 0).double().mean()))
    return dict(G=G, b2=b2, out=out, out_pm=out.float().half().transpose(1, 2).contiguous(), stats=stats)


# ---- pm_linear ----------------------------------------------------------------------------------------------------
PM_HIDDEN, PM_OUT_CM, PM_OUT_PM32, PM_VOTE, PM_LINEAR = 0, 1, 2, 3, 4     # _ext.PM_* (importable without torch CUDA)
PM_NAMES = {PM_HIDDEN: "HIDDEN", PM_OUT_CM: "OUT_CM", PM_OUT_PM32: "OUT_PM32", PM_VOTE: "VOTE", PM_LINEAR: "LINEAR"}
# (mode, M, points_per_scene, K, N, lo, want_lo): lo = "x" -> X is an fp16 pair with non-zero lo parts and W is
# fp16-exact; "w" -> X is plain fp16 (no lo operand) and W has non-zero lo parts
PM_CASES = [
    (PM_HIDDEN, 4096, 1024, 512, 256, "w", True), (PM_HIDDEN, 647, 647, 136, 96, "x", True),
    (PM_HIDDEN, 1, 1, 64, 32, "w", False),
    (PM_OUT_CM, 647, 647, 264, 256, "x", True), (PM_OUT_CM, 127, 127, 8, 32, "w", False),
    (PM_OUT_CM, 4096, 512, 64, 96, "x", True),
    (PM_OUT_PM32, 127, 127, 64, 5, "w", True), (PM_OUT_PM32, 647, 647, 512, 79, "x", True),
    (PM_OUT_PM32, 4096, 1024, 136, 272, "w", True), (PM_OUT_PM32, 1, 1, 8, 272, "x", True),
    (PM_LINEAR, 4096, 2048, 264, 96, "x", False), (PM_LINEAR, 647, 647, 8, 256, "w", True),
    (PM_LINEAR, 127, 127, 512, 32, "x", False),
    (PM_VOTE, 647, 647, 256, 259, "w", True), (PM_VOTE, 4096, 1024, 64, 35, "x", False),
    (PM_VOTE, 127, 127, 136, 99, "x", True),
]
# launch hints (pm_n_tile, pm_tiles_per_cta): channel slices of 16 .. 256 (16 and 48: a slice that is not a whole
# number of 32-channel blocks), one to sixteen row tiles per CTA
PM_HINTS = ((0, 0), (16, 2), (48, 0), (64, 3), (256, 4), (128, 16))


def _pm_id(c):
    mode, M, n, K, N, lo, want_lo = c
    return "%s-M%d-K%d-N%d-%slo%s" % (PM_NAMES[mode], M, K, N, lo, "" if want_lo else "-nolo")


def make_pm_case(mode, M, n, K, N, lo, want_lo, seed=0):
    rng = np.random.default_rng([seed, mode, M, K, N])
    R = max(1, 512 // K)                              # integer operands in [-R, R]: K * R * 2^12 <= 2^21
    ints = lambda shape: rng.integers(-R, R + 1, size=shape).astype(np.float64)                          # noqa: E731
    # +-m * 2^-12, m in [2048, 4096): 12 significant bits, i.e. an fp16 hi and a lo of 0 or +-2^-12
    frac = lambda shape: rng.choice([-1.0, 1.0], size=shape) * rng.integers(2048, 4096, size=shape) * 2.0 ** -12  # noqa
    x, W = (ints((M, K)), frac((N, K))) if lo == "w" else (frac((M, K)), ints((N, K)))
    c = dict(mode=mode, M=M, n=n, K=K, N=N, lo=lo, want_lo=want_lo, x=x, W=W,
             b=rng.integers(-R * 4096, R * 4096 + 1, size=N) * 2.0 ** -12)
    if mode == PM_VOTE:
        B, D = M // n, N - 3
        c["seed_cm"] = rng.integers(-R * 4096, R * 4096 + 1, size=(B, D, n)) * 2.0 ** -12
        c["seed_xyz"] = rng.integers(-R * 4096, R * 4096 + 1, size=(B, n, 3)) * 2.0 ** -12
    return c


def pm_reference(c):
    """float64 result of the layer (numpy), and the preconditions."""
    T = lambda a: torch.as_tensor(a, dtype=torch.float64)        # noqa: E731
    x, W, b = T(c["x"]), T(c["W"]), T(c["b"])
    (xh, xl), (wh, wl) = _split16(x), _split16(W)
    if c["lo"] == "w":
        assert torch.equal(xl, torch.zeros_like(xl)) and bool((wl != 0).any())
    else:
        assert torch.equal(wl, torch.zeros_like(wl)) and bool((xl != 0).any())
    budget = _Budget()
    extra = 0.0
    if c["mode"] == PM_VOTE:
        extra = max(float(np.abs(c["seed_cm"]).max()), float(np.abs(c["seed_xyz"]).max()))
    budget.add("x.W^T + b", (xh.abs() + xl.abs()) @ wh.abs().t() + xh.abs() @ wl.abs().t() + b.abs() + extra,
               max(_q(xh) + _q(wh), _q(xl) + _q(wh), _q(xh) + _q(wl), _q(b), 12))
    budget.check()
    v = x @ W.t() + b                                            # (M, N)
    r = dict(v=v)
    M, n, N = c["M"], c["n"], c["N"]
    if c["mode"] == PM_VOTE:
        B, D = M // n, N - 3
        f = T(c["seed_cm"]).transpose(1, 2).reshape(M, D) + v[:, :D]
        r["vote_xyz"] = T(c["seed_xyz"]) + v[:, D:].reshape(B, n, 3)
        r["f"] = f
        r["out"] = (f / f.norm(dim=1, keepdim=True)).view(B, n, D).transpose(1, 2)
        assert _is_f32(f) and _is_f32(r["vote_xyz"])
        return r
    y = torch.relu(v) if c["mode"] in (PM_HIDDEN, PM_OUT_CM) else v
    assert _is_f32(y)
    hi, lo = _split16(y)                                         # the exact result is an exact fp16 pair
    assert torch.equal(hi + lo, y)
    r.update(y=y, hi=hi, lo=lo)
    if c["mode"] == PM_OUT_CM:
        r["out"] = y.view(M // n, n, N).transpose(1, 2)
    return r


# ---- interp_cat_pm and three_nn_weights -----------------------------------------------------------------------------
INTERP_CASES = [(8, 0, 77), (256, 8, 1001), (264, 256, 333), (8, 256, 1)]       # (C2, C1, n)
NN_CASES = [3, 5, 1500, 3000]                                                    # m


def make_nn_case(m, B=3, n=333, seed=0):
    """Lattice clouds: known points on a small integer lattice (duplicates and exact distance ties), unknown points
    that are known points (zero distances), lattice points and half-integer points (more ties)."""
    rng = np.random.default_rng([seed, m])
    L = max(2, int(round(m ** (1 / 3))))
    known = rng.integers(0, L, size=(B, m, 3)).astype(np.float32)
    unknown = rng.integers(-1, L + 1, size=(B, n, 3)).astype(np.float32)
    unknown[:, 1::3] += 0.5
    pick = rng.integers(0, m, size=(B, n // 3))
    unknown[:, 2::3][:, :n // 3] = known[np.arange(B)[:, None], pick][:, :unknown[:, 2::3].shape[1]]
    return unknown, known


def nn_weights_reference(unknown, known):
    """oracle.three_nn + the kernel's formula in numpy float32: 1 / (sqrt(d) + 1e-8), left-to-right sum, divide."""
    import oracle
    d2, idx = oracle.three_nn(unknown, known)
    r = np.float32(1) / (np.sqrt(d2) + np.float32(1e-8))
    norm = (r[..., 0] + r[..., 1]) + r[..., 2]
    return idx, r / norm[..., None]


# =================================================================================================================
def test_generators_meet_preconditions():
    """Every case of this file, in float64 on the CPU: all intermediates on their storage grids, every partial sum
    inside the accumulator margin, the fp16 splits exact, both lo operands exercised, the ReLUs clipping."""
    seen_lo = set()
    for case in SA_CASES:
        c = make_sa_case(*case)
        r = sa_reference(c, "cpu")
        st = r["stats"]
        for k in ("relu0", "relu1", "relu2"):
            assert 0.05 < st[k] < 0.95, (case, k, st[k])
        if c["form"] == "inline":
            lo = case[6]
            # (without features there is nothing to cancel against: Cf = 0 runs the xyz inputs only)
            assert st["x_lo"] == st["b_lo"] == (lo == "x" and c["Cf"] > 0)
            assert st["w_lo"] == (lo == "w")
            seen_lo |= {k for k in ("x_lo", "w_lo", "b_lo") if st[k]}
    assert seen_lo == {"x_lo", "w_lo", "b_lo"}
    widths = {case[1:5] for case in SA_CASES if case[0] == "inline"}
    assert len(widths) == 9 and {case[1:5] for case in SA_CASES if case[0] == "proj"} == widths
    for case in PM_CASES:
        pm_reference(make_pm_case(*case))
    assert {case[0] for case in PM_CASES} == set(PM_NAMES)


# =================================================================================================================
def _cu(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a)).to(device=DEV, dtype=dtype).contiguous()


def _mismatch(got, want):
    got, want = got.double().cpu(), want.double().cpu()
    bad = got != want
    if not bool(bad.any()):
        return ""
    i = int(bad.flatten().nonzero()[0])
    return "%d of %d differ, first at flat index %d: %r != %r" % (int(bad.sum()), bad.numel(), i,
                                                                  float(got.flatten()[i]), float(want.flatten()[i]))


@pytest.mark.gpu
@pytest.mark.parametrize("case", SA_CASES, ids=[_sa_id(c) for c in SA_CASES])
def test_sa_fused_exact(case):
    """_ext.sa_fused_forward with explicit weights == the float64 evaluation, bit for bit, under every sa_min_tiles
    hint; the point-major fp16 copy == the fp16 rounding of the fp32 output."""
    from spacap3d_b200 import _ext
    c = make_sa_case(*case)
    ref = sa_reference(c, DEV)
    H = _ext.HALF
    xyz, new_xyz, idx = _cu(c["xyz"]), _cu(c["new_xyz"]), _cu(c["idx"], torch.int32)
    W0, b0, W1, W2 = _cu(c["W0"]), _cu(c["b0"]), _cu(c["W1"], H), _cu(c["W2"], H)
    b1, b2 = _cu(c["b1"]), ref["b2"].float().contiguous()
    kw = dict(radius=c["radius"], want_point_major=True)
    if c["form"] == "inline":
        kw["feat"] = _cu(c["feat"]) if c["Cf"] else None
    else:
        Wf = _ext.split_half(_cu(c["W0f"]))
        G, G_lo = _ext.pm_linear(_cu(c["feat_pm"], H), Wf, torch.zeros(c["C1"], device=DEV), _ext.PM_LINEAR,
                                 c["n"], want_lo=False)
        assert G_lo is None
        assert torch.equal(G.double(), ref["G"]), _mismatch(G, ref["G"])
        kw["G"] = G.view(c["B"], c["n"], c["C1"])
    for hint in SA_MIN_TILES:
        with _ext.launch_options(sa_min_tiles=hint):
            out, out_pm = _ext.sa_fused_forward(xyz, new_xyz, idx, W0, b0, W1, b1, W2, b2, **kw)
        assert torch.equal(out.double(), ref["out"]), (hint, _mismatch(out, ref["out"]))
        assert torch.equal(out_pm, out.transpose(1, 2).half()), (hint, _mismatch(out_pm, out.transpose(1, 2)))
        assert torch.equal(out_pm, ref["out_pm"]), hint


@pytest.mark.gpu
@pytest.mark.parametrize("case", PM_CASES, ids=[_pm_id(c) for c in PM_CASES])
def test_pm_linear_exact(case):
    """Every pm_linear mode == the float64 evaluation: the fp16 pair and the fp32 outputs bit for bit (the vote tail's
    L2-normalised outputs within the bound of its fp32 arithmetic), under every launch hint."""
    from spacap3d_b200 import _ext
    c = make_pm_case(*case)
    ref = pm_reference(c)
    mode, M, n, N, want_lo = c["mode"], c["M"], c["n"], c["N"], c["want_lo"]
    X = _ext.split_half(_cu(c["x"])) if c["lo"] == "x" else _cu(c["x"], _ext.HALF)
    W, b = _ext.split_half(_cu(c["W"])), _cu(c["b"])
    if c["lo"] == "x":
        assert bool((X[1] != 0).any())
    else:
        assert bool((W[1] != 0).any())
    kw = dict(want_lo=want_lo)
    if mode == PM_VOTE:
        kw.update(seed_cm=_cu(c["seed_cm"]), seed_xyz=_cu(c["seed_xyz"]))
    for hint in PM_HINTS:
        with _ext.launch_options(pm_n_tile=hint[0], pm_tiles_per_cta=hint[1]):
            res = _ext.pm_linear(X, W, b, mode, n, **kw)
        if mode == PM_OUT_PM32:
            assert torch.equal(res.double().cpu(), ref["v"]), (hint, _mismatch(res, ref["v"]))
            continue
        if mode in (PM_HIDDEN, PM_LINEAR):
            hi, lo = res
        elif mode == PM_OUT_CM:
            out, (hi, lo) = res
            assert torch.equal(out.double().cpu(), ref["out"]), (hint, _mismatch(out, ref["out"]))
        else:
            vote_xyz, out, (hi, lo) = res
            assert torch.equal(vote_xyz.double().cpu(), ref["vote_xyz"]), (hint, _mismatch(vote_xyz, ref["vote_xyz"]))
            # The pair is the kernel's own fp32 result split by split_f16: exactly reproducible from `out`.
            pm = out.transpose(1, 2).reshape(M, N - 3)
            assert torch.equal(hi, pm.half()), hint
            if want_lo:
                assert torch.equal(lo, (pm - hi.float()).half()), hint
            # out = f / ||f|| from exact f, in fp32 (u = 2^-24): the D fmaf steps of the squared norm, all terms
            # non-negative, give s(1 + t) with |t| <= gamma_D = D u / (1 - D u); sqrtf, the division 1/x and the
            # product f * inv are correctly rounded (IEEE, no fast-math), one factor (1 + d), |d| <= u, each.  So
            # |out - f/||f||| <= |f/||f||| ((1 - gamma_D)^(-1/2) (1 + u)^2 / (1 - u) - 1), element by element.
            u, D = 2.0 ** -24, N - 3
            gamma = D * u / (1 - D * u)
            rel = (1 - gamma) ** -0.5 * (1 + u) ** 2 / (1 - u) - 1
            err = (out.double().cpu() - ref["out"]).abs()
            assert bool((err <= ref["out"].abs() * rel).all()), (hint, float((err / ref["out"].abs()).max()), rel)
            assert (lo is None) == (not want_lo)
            continue
        assert torch.equal(hi.double().cpu(), ref["hi"]), (hint, _mismatch(hi, ref["hi"]))
        assert (lo is None) == (not want_lo)
        if want_lo:
            assert torch.equal(hi.double().cpu() + lo.double().cpu(), ref["y"]), (hint, _mismatch(lo, ref["lo"]))


@pytest.mark.gpu
@pytest.mark.parametrize("C2,C1,n", INTERP_CASES)
def test_interp_cat_pm_exact(C2, C1, n):
    """interp_cat_pm == oracle.three_interpolate (the same fmaf order) on the fp16 rows widened to fp32, rounded to
    fp16 (round to nearest even), followed by the skip rows, bit for bit."""
    import oracle
    from spacap3d_b200 import _ext
    rng = np.random.default_rng([C2, C1, n])
    B, m = 3, 300
    known = rng.standard_normal((B, m, C2)).astype(np.float16)
    skip = rng.standard_normal((B, n, C1)).astype(np.float16)
    idx = rng.integers(0, m, size=(B, n, 3)).astype(np.int32)
    idx[:, ::7, 1] = idx[:, ::7, 0]                               # repeated neighbours
    idx[:, 0] = [0, m - 1, m - 1]
    w = rng.random((B, n, 3)).astype(np.float32)
    w[:, ::5, 2] = 0
    w = w / w.sum(-1, keepdims=True, dtype=np.float32)
    got = _ext.interp_cat_pm(_cu(known, _ext.HALF), _cu(idx, torch.int32), _cu(w), _cu(skip, _ext.HALF))
    interp = oracle.three_interpolate(known.astype(np.float32).transpose(0, 2, 1), idx, w)      # (B,C2,n) f32
    want = np.concatenate([interp.transpose(0, 2, 1).astype(np.float16), skip], -1)
    got = got.cpu().numpy()
    assert got.shape == want.shape
    np.testing.assert_array_equal(got.view(np.uint16), want.view(np.uint16))


@pytest.mark.gpu
@pytest.mark.parametrize("m", NN_CASES)
def test_three_nn_weights_exact(m):
    """three_nn_weights: idx == oracle.three_nn (ties go to the lower index) and the weights bit for bit equal to the
    same formula in numpy float32, on lattice clouds with exact ties, duplicated points and zero distances; m = 1500
    and 3000 span several 1024-point shared-memory tiles."""
    from spacap3d_b200 import _ext
    unknown, known = make_nn_case(m)
    idx, w = _ext.three_nn_weights(_cu(unknown), _cu(known))
    want_idx, want_w = nn_weights_reference(unknown, known)
    np.testing.assert_array_equal(idx.cpu().numpy(), want_idx)
    np.testing.assert_array_equal(w.cpu().numpy().view(np.uint32), want_w.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("npoint,nsample", [(64, 8), (100, 16)])
def test_unfused_fallback(npoint, nsample):
    """A layer without a fused kernel (nsample 8; npoint * nsample not a multiple of 128) warns once with a
    RuntimeWarning and returns exactly what the reference op sequence (FAST_PATHS = False) returns."""
    from spacap3d_b200 import pointnet2_modules as M
    from spacap3d_b200.scenes import make_scene_xyz
    torch.manual_seed(0)
    m = M.PointnetSAModuleVotes(npoint=npoint, radius=0.3, nsample=nsample, mlp=[1, 64, 64, 128], use_xyz=True,
                                normalize_xyz=True).to(DEV).eval()
    xyz = torch.from_numpy(np.stack([make_scene_xyz(5 + i, 2048) for i in range(3)], 0)).to(DEV)
    feats = torch.randn(3, 1, 2048, generator=torch.Generator().manual_seed(1)).to(DEV)
    old = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        with torch.no_grad(), warnings.catch_warnings(record=True) as rec:
            warnings.simplefilter("always")
            got = [m(xyz, feats) for _ in range(2)]
            M.FAST_PATHS = False
            want = m(xyz, feats)
    finally:
        M.FAST_PATHS = True
        torch.backends.cudnn.deterministic = old
    unfused = [r for r in rec if issubclass(r.category, RuntimeWarning) and "no fused set-abstraction" in str(r.message)]
    assert len(unfused) == 1, [str(r.message) for r in rec]
    for g in got:
        assert all(torch.equal(a, b) for a, b in zip(g, want))
