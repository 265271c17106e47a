"""Drop-in for the reference's pybind11 module `pointnet2._ext`
(lib/pointnet2/_ext_src/src/bindings.cpp:6-19): the same nine callables with the same argument
order, dtype/contiguity/device checks (include/utils.h:5-25 -> RuntimeError) and return values,
implemented by libspacap3d_ops.so through its C ABI (include/spacap3d_ops.h).

Differences, all invisible to callers: outputs are allocated with torch.empty (every element is
written by the kernels), launches go to torch's *current* stream under a device guard taken from
the input tensor, and a failed launch raises instead of calling exit(-1).
"""
import math
import threading

import torch

from . import _lib

# 16-bit storage type of the eval fast paths (fused SA operands, point-major activations).  fp16, not bf16: 11
# significant bits instead of 8 at the same tensor-core rate, ~8x closer to the fp32 reference; the kernels saturate
# at +-65504 instead of overflowing (csrc/sa_fused.cu).
HALF = torch.float16


def _check(t, name, dtype):
    if not isinstance(t, torch.Tensor):
        raise RuntimeError("%s must be a tensor" % name)
    if not t.is_contiguous():
        raise RuntimeError("%s must be a contiguous tensor" % name)
    if t.dtype != dtype:
        kind = {torch.float32: "a float", torch.int32: "an int"}.get(dtype, "a " + str(dtype))
        raise RuntimeError("%s must be %s tensor" % (name, kind))


def _storage(t, name):
    """Entry-point suffix of a tensor the training-path kernels store as fp32 ('') or bf16 ('_bf16': the
    torch.autocast(dtype=torch.bfloat16) twins).  Any other dtype raises the fp32 check's message."""
    if isinstance(t, torch.Tensor) and t.dtype == torch.bfloat16:
        _check(t, name, torch.bfloat16)
        return "_bf16"
    _check(t, name, torch.float32)
    return ""


def _grad_as(grad, t):
    """The bf16 twins write fp32 gradients (no bf16 atomics); autograd wants them in the dtype of the forward input,
    which is that of the incoming gradient t: one rounding."""
    return grad if t.dtype == grad.dtype else grad.to(t.dtype)


def _same_device(a, *rest):
    """Checked after dtype/contiguity of every argument, like the reference (sampling.cpp:15-35)."""
    if not a.is_cuda:
        raise RuntimeError("CPU not supported")  # sampling.cpp:33-35 etc.
    for t in rest:
        if not t.is_cuda:
            raise RuntimeError("all tensors must be CUDA tensors")
        if t.device != a.device:
            raise RuntimeError("all tensors must be on the same CUDA device")


def _stream():
    return torch.cuda.current_stream().cuda_stream


# clouds at least this large get a workspace, which lets the library use its bucketed FPS kernel
# (fps.cu); the result is identical either way
FPS_WORKSPACE_MIN_N = 4096

FPS_AUTO, FPS_CLUSTER, FPS_BUCKET = 0, 1, 2      # include/spacap3d_ops.h SPC_FPS_*
FPS_BUCKET_MIN_N, FPS_BUCKET_MAX_N = 4096, 40960  # size range of the bucketed sampler


class _LaunchOptions(threading.local):
    """Per-THREAD launch hints handed to the library with every call (the C ABI keeps no mutable state, so that
    nn.DataParallel worker threads / several pipelines in one process cannot disturb each other).  None of them
    changes results."""
    fps_algo = FPS_AUTO        # sampler selection for large clouds
    sa_min_tiles = 0           # fused SA kernel: at least this many 128-row tiles per CTA (0 = one CTA per SM)
    pm_n_tile = 0              # pm_linear: output channels per CTA (0 = 128: lowest latency; 256 = fewest CTAs)
    pm_tiles_per_cta = 0       # pm_linear: 128-row tiles per CTA (0 = 1; > 1: double-buffered accumulator, fewer CTAs)


_options = _LaunchOptions()


class launch_options:
    """Context manager: `with launch_options(sa_min_tiles=16): ...` (thread-local, re-entrant)."""

    def __init__(self, **kw):
        for k in kw:
            if not hasattr(_LaunchOptions, k):
                raise TypeError("unknown launch option %r" % k)
        self.kw = kw

    def __enter__(self):
        self.saved = {k: getattr(_options, k) for k in self.kw}
        for k, v in self.kw.items():
            setattr(_options, k, v)
        return self

    def __exit__(self, *exc):
        for k, v in self.saved.items():
            setattr(_options, k, v)


def _fps_algo(N):
    """The thread's sampler preference for a cloud of N points: a preference for the bucketed sampler only applies
    inside its size range (a forward samples clouds of 40 000, 2 048, 1 024 ... points under one setting)."""
    a = int(_options.fps_algo)
    if a == FPS_BUCKET and not FPS_BUCKET_MIN_N <= N <= FPS_BUCKET_MAX_N:
        return FPS_AUTO
    return a


def furthest_point_sampling(points, nsamples):
    """(B,N,3) f32 -> (B,nsamples) i32.   sampling.cpp:66-87"""
    _check(points, "points", torch.float32)
    _same_device(points)
    B, N, _ = points.shape
    out = torch.empty((B, nsamples), dtype=torch.int32, device=points.device)
    with torch.cuda.device(points.device):
        if N >= FPS_WORKSPACE_MIN_N and nsamples >= 2:
            nbytes = _lib.load().spc_fps_workspace_bytes(B, N, int(nsamples))
            ws = torch.empty((nbytes + 3) // 4, dtype=torch.int32, device=points.device)
            _lib.call("spc_furthest_point_sampling_ex2", points.data_ptr(), B, N, int(nsamples),
                      out.data_ptr(), None, 0, None, None, ws.data_ptr(), nbytes, _fps_algo(N), _stream())
        else:
            _lib.call("spc_furthest_point_sampling", points.data_ptr(), B, N, int(nsamples),
                      out.data_ptr(), None, _stream())
    return out


def furthest_point_sampling_with_xyz(points, nsamples, hint_ordered=False, known_ordered=None, want_strict=False):
    """Extension: FPS that also returns the sampled coordinates (B,nsamples,3) from the same
    kernel (the gather that always follows FPS, pointnet2_modules.py:237-242).

    hint_ordered=True tells the library that `points` is probably itself an FPS output (SA2..SA4
    sample from the previous layer's centres); it then PROVES, with two parallel kernels, whether
    the result is 0..nsamples-1 and skips the sequential rounds for the scenes where it is.  The
    returned indices are identical with or without the hint (spc_furthest_point_sampling_ex).

    want_strict=True additionally returns a (B,) int32 device tensor: 1 = every pick was the strict unique
    maximum, i.e. the OUTPUT is a strict FPS sequence; passing it as `known_ordered` to the call that samples
    from that output skips proof and rounds for the flagged scenes (spc_furthest_point_sampling_ex2)."""
    _check(points, "points", torch.float32)
    _same_device(points)
    B, N, _ = points.shape
    out = torch.empty((B, nsamples), dtype=torch.int32, device=points.device)
    new_xyz = torch.empty((B, nsamples, 3), dtype=torch.float32, device=points.device)
    if want_strict or known_ordered is not None:
        strict = torch.empty(B, dtype=torch.int32, device=points.device) if want_strict else None
        if known_ordered is not None:
            _check(known_ordered, "known_ordered", torch.int32)
            assert known_ordered.numel() == B and nsamples <= N
        with torch.cuda.device(points.device):
            nbytes = _lib.load().spc_fps_workspace_bytes(B, N, int(nsamples))
            ws = torch.empty((nbytes + 3) // 4, dtype=torch.int32, device=points.device)
            _lib.call("spc_furthest_point_sampling_ex2", points.data_ptr(), B, N, int(nsamples), out.data_ptr(),
                      new_xyz.data_ptr(), int(bool(hint_ordered) and 2 <= nsamples <= N),
                      known_ordered.data_ptr() if known_ordered is not None else None,
                      strict.data_ptr() if strict is not None else None, ws.data_ptr(), nbytes,
                      _fps_algo(N), _stream())
        return (out, new_xyz, strict) if want_strict else (out, new_xyz)
    with torch.cuda.device(points.device):
        if (hint_ordered and 2 <= nsamples <= N) or (N >= FPS_WORKSPACE_MIN_N and nsamples >= 2):
            nbytes = _lib.load().spc_fps_workspace_bytes(B, N, int(nsamples))
            ws = torch.empty((nbytes + 3) // 4, dtype=torch.int32, device=points.device)
            _lib.call("spc_furthest_point_sampling_ex2", points.data_ptr(), B, N, int(nsamples),
                      out.data_ptr(), new_xyz.data_ptr(), int(bool(hint_ordered)), None, None, ws.data_ptr(), nbytes,
                      _fps_algo(N), _stream())
        else:
            _lib.call("spc_furthest_point_sampling", points.data_ptr(), B, N, int(nsamples),
                      out.data_ptr(), new_xyz.data_ptr(), _stream())
    return out, new_xyz


def gather_points(points, idx):
    """(B,C,N), (B,M) -> (B,C,M).   sampling.cpp:15-38"""
    _check(points, "points", torch.float32)
    _check(idx, "idx", torch.int32)
    _same_device(points, idx)
    B, C, N = points.shape
    M = idx.shape[1]
    out = torch.empty((B, C, M), dtype=torch.float32, device=points.device)
    with torch.cuda.device(points.device):
        _lib.call("spc_gather_points", points.data_ptr(), idx.data_ptr(), B, C, N, M,
                  out.data_ptr(), _stream())
    return out


def gather_points_grad(grad_out, idx, n):
    """(B,C,M), (B,M) -> (B,C,n).   sampling.cpp:40-65"""
    _check(grad_out, "grad_out", torch.float32)
    _check(idx, "idx", torch.int32)
    _same_device(grad_out, idx)
    B, C, M = grad_out.shape
    out = torch.empty((B, C, int(n)), dtype=torch.float32, device=grad_out.device)
    with torch.cuda.device(grad_out.device):
        _lib.call("spc_gather_points_grad", grad_out.data_ptr(), idx.data_ptr(), B, C, int(n), M,
                  out.data_ptr(), _stream())
    return out


def ball_query(new_xyz, xyz, radius, nsample):
    """(B,M,3), (B,N,3) -> (B,M,nsample) i32.   ball_query.cpp:8-32"""
    _check(new_xyz, "new_xyz", torch.float32)
    _check(xyz, "xyz", torch.float32)
    _same_device(new_xyz, xyz)
    B, M, _ = new_xyz.shape
    N = xyz.shape[1]
    out = torch.empty((B, M, int(nsample)), dtype=torch.int32, device=new_xyz.device)
    with torch.cuda.device(new_xyz.device):
        if N >= 1024:      # uniform-grid search (bit-identical output); tiny clouds stay all-pairs
            nbytes = _lib.load().spc_ball_query_workspace_bytes(B, N)
            ws = torch.empty((nbytes + 3) // 4, dtype=torch.int32, device=new_xyz.device)
            _lib.call("spc_ball_query_ex", new_xyz.data_ptr(), xyz.data_ptr(), B, N, M, float(radius),
                      int(nsample), out.data_ptr(), ws.data_ptr(), nbytes, _stream())
        else:
            _lib.call("spc_ball_query", new_xyz.data_ptr(), xyz.data_ptr(), B, N, M, float(radius),
                      int(nsample), out.data_ptr(), _stream())
    return out


def group_points(points, idx):
    """(B,C,N), (B,npoint,nsample) -> (B,C,npoint,nsample), f32 or bf16 like points.   group_points.cpp:12-36"""
    sfx = _storage(points, "points")
    _check(idx, "idx", torch.int32)
    _same_device(points, idx)
    B, C, N = points.shape
    _, npoint, nsample = idx.shape
    out = torch.empty((B, C, npoint, nsample), dtype=points.dtype, device=points.device)
    with torch.cuda.device(points.device):
        _lib.call("spc_group_points" + sfx, points.data_ptr(), idx.data_ptr(), B, C, N, npoint, nsample,
                  out.data_ptr(), _stream())
    return out


def group_points_grad(grad_out, idx, n):
    """(B,C,npoint,nsample), (B,npoint,nsample) -> (B,C,n) in grad_out's dtype (f32 or bf16; accumulated in
    fp32).   group_points.cpp:38-62"""
    sfx = _storage(grad_out, "grad_out")
    _check(idx, "idx", torch.int32)
    _same_device(grad_out, idx)
    B, C, npoint, nsample = grad_out.shape
    out = torch.empty((B, C, int(n)), dtype=torch.float32, device=grad_out.device)
    with torch.cuda.device(grad_out.device):
        nbytes = _lib.load().spc_group_points_grad_workspace_bytes(B, int(n), npoint, nsample) if C >= 4 else 0
        if nbytes:
            ws = torch.empty((nbytes + 3) // 4, dtype=torch.int32, device=grad_out.device)
            _lib.call("spc_group_points_grad_ex" + sfx, grad_out.data_ptr(), idx.data_ptr(), B, C, int(n),
                      npoint, nsample, out.data_ptr(), ws.data_ptr(), nbytes, _stream())
        else:
            _lib.call("spc_group_points_grad" + sfx, grad_out.data_ptr(), idx.data_ptr(), B, C, int(n),
                      npoint, nsample, out.data_ptr(), _stream())
    return _grad_as(out, grad_out)


def three_nn(unknowns, knows):
    """(B,n,3), (B,m,3) -> [dist2 (B,n,3) f32, idx (B,n,3) i32].   interpolate.cpp:14-40"""
    _check(unknowns, "unknowns", torch.float32)
    _check(knows, "knows", torch.float32)
    _same_device(unknowns, knows)
    B, n, _ = unknowns.shape
    m = knows.shape[1]
    dist2 = torch.empty((B, n, 3), dtype=torch.float32, device=unknowns.device)
    idx = torch.empty((B, n, 3), dtype=torch.int32, device=unknowns.device)
    with torch.cuda.device(unknowns.device):
        _lib.call("spc_three_nn", unknowns.data_ptr(), knows.data_ptr(), B, n, m,
                  dist2.data_ptr(), idx.data_ptr(), _stream())
    return [dist2, idx]


def three_interpolate(points, idx, weight):
    """(B,C,m), (B,n,3), (B,n,3) f32 -> (B,C,n), f32 or bf16 like points.   interpolate.cpp:42-70"""
    sfx = _storage(points, "points")
    _check(idx, "idx", torch.int32)
    _check(weight, "weight", torch.float32)
    _same_device(points, idx, weight)
    B, C, m = points.shape
    n = idx.shape[1]
    out = torch.empty((B, C, n), dtype=points.dtype, device=points.device)
    with torch.cuda.device(points.device):
        _lib.call("spc_three_interpolate" + sfx, points.data_ptr(), idx.data_ptr(), weight.data_ptr(),
                  B, C, m, n, out.data_ptr(), _stream())
    return out


def three_interpolate_grad(grad_out, idx, weight, m):
    """(B,C,n), (B,n,3), (B,n,3) f32 -> (B,C,m) in grad_out's dtype (f32 or bf16; accumulated in fp32).
    interpolate.cpp:71-99"""
    sfx = _storage(grad_out, "grad_out")
    _check(idx, "idx", torch.int32)
    _check(weight, "weight", torch.float32)
    _same_device(grad_out, idx, weight)
    B, C, n = grad_out.shape
    out = torch.empty((B, C, int(m)), dtype=torch.float32, device=grad_out.device)
    with torch.cuda.device(grad_out.device):
        _lib.call("spc_three_interpolate_grad" + sfx, grad_out.data_ptr(), idx.data_ptr(),
                  weight.data_ptr(), B, C, n, int(m), out.data_ptr(), _stream())
    return _grad_as(out, grad_out)


def sa_fused_forward(xyz, new_xyz, idx, W0, b0, W1, b1, W2, b2, *, G=None, feat=None, radius=1.0,
                     want_point_major=False):
    """Fused set-abstraction forward (eval): gather + layer 0 + two tcgen05 1x1 convs + max-pool.
    See spc_sa_fused_forward in include/spacap3d_ops.h.
      in-line form   : G is None, feat (B,Cf,n) or None, W0 (C1,3+Cf)
      projected form : G (B,n,C1) fp16 = per-point projection of the features, W0 (C1,3)
    Returns out (B,C3,npoint) f32, and also the point-major fp16 copy (B,npoint,C3) when
    want_point_major.  Raises _lib.SpcUnsupported when the library has no kernel for the shape
    (the caller then uses the unfused CUDA ops)."""
    _check(xyz, "xyz", torch.float32)
    _check(new_xyz, "new_xyz", torch.float32)
    _check(idx, "idx", torch.int32)
    _check(W0, "W0", torch.float32)
    _check(b0, "b0", torch.float32)
    _check(W1, "W1", HALF)
    _check(W2, "W2", HALF)
    _check(b1, "b1", torch.float32)
    _check(b2, "b2", torch.float32)
    _same_device(xyz, new_xyz, idx, W0, b0, W1, b1, W2, b2)
    B, n, _ = xyz.shape
    _, npoint, nsample = idx.shape
    C2, C1 = W1.shape
    C3 = W2.shape[0]
    assert W2.shape[1] == C2 and b1.numel() == C2 and b2.numel() == C3 and b0.numel() == C1
    Cf, pG, pfeat = 0, None, None
    if G is not None:
        _check(G, "G", HALF)
        _same_device(xyz, G)
        assert G.shape == (B, n, C1) and W0.shape == (C1, 3)
        pG = G.data_ptr()
    else:
        if feat is not None:
            _check(feat, "feat", torch.float32)
            _same_device(xyz, feat)
            Cf = feat.shape[1]
            pfeat = feat.data_ptr()
        assert W0.shape == (C1, 3 + Cf)
    out = torch.empty((B, C3, npoint), dtype=torch.float32, device=xyz.device)
    out_pm = torch.empty((B, npoint, C3), dtype=HALF, device=xyz.device) if want_point_major else None
    with torch.cuda.device(xyz.device):
        # the two None after b0 fill the W0_host / b0_host slots, which the library ignores
        _lib.call("spc_sa_fused_forward_ex", xyz.data_ptr(), new_xyz.data_ptr(), idx.data_ptr(),
                  pG, pfeat, W0.data_ptr(), b0.data_ptr(), None, None, int(Cf), float(radius), W1.data_ptr(),
                  b1.data_ptr(), W2.data_ptr(), b2.data_ptr(), B, n, npoint, nsample, C1, C2, C3,
                  out.data_ptr(), out_pm.data_ptr() if out_pm is not None else None, int(_options.sa_min_tiles),
                  _stream())
    return (out, out_pm) if want_point_major else out


def three_nn_weights(unknown, known):
    """three_nn + normalised inverse-distance weights in one kernel -> (idx (B,n,3) i32, weight (B,n,3) f32)
    (pointnet2_modules.py:398-402)."""
    _check(unknown, "unknown", torch.float32)
    _check(known, "known", torch.float32)
    _same_device(unknown, known)
    B, n, _ = unknown.shape
    m = known.shape[1]
    idx = torch.empty((B, n, 3), dtype=torch.int32, device=unknown.device)
    w = torch.empty((B, n, 3), dtype=torch.float32, device=unknown.device)
    with torch.cuda.device(unknown.device):
        _lib.call("spc_three_nn_weights", unknown.data_ptr(), known.data_ptr(), B, n, m, idx.data_ptr(),
                  w.data_ptr(), _stream())
    return idx, w


def interp_cat_pm(known_pm, idx, weight, skip_pm):
    """Point-major fp16: X (B,n,C2+C1) = [3-NN interpolation of known_pm (B,m,C2), skip_pm (B,n,C1)]."""
    _check(known_pm, "known_pm", HALF)
    _check(idx, "idx", torch.int32)
    _check(weight, "weight", torch.float32)
    _check(skip_pm, "skip_pm", HALF)
    _same_device(known_pm, idx, weight, skip_pm)
    B, m, C2 = known_pm.shape
    n, C1 = skip_pm.shape[1], skip_pm.shape[2]
    X = torch.empty((B, n, C2 + C1), dtype=HALF, device=known_pm.device)
    with torch.cuda.device(known_pm.device):
        _lib.call("spc_interp_cat_pm", known_pm.data_ptr(), idx.data_ptr(), weight.data_ptr(), skip_pm.data_ptr(),
                  B, n, m, C2, C1, X.data_ptr(), _stream())
    return X


PM_HIDDEN, PM_OUT_CM, PM_OUT_PM32, PM_VOTE, PM_LINEAR = 0, 1, 2, 3, 4     # include/spacap3d_ops.h SPC_PM_*


def split_half(w):
    """fp32 tensor -> (hi, lo) fp16 pair with w ~= hi + lo to ~2^-22 (operands of spc_pm_linear)."""
    hi = w.to(HALF)
    lo = (w - hi.float()).to(HALF)
    return hi.contiguous(), lo.contiguous()


def pm_linear(X, W, bias, mode, points_per_scene, seed_cm=None, seed_xyz=None, want_lo=True):
    """One point-major 1x1-conv layer on tcgen05 (spc_pm_linear).  X: (M,K) fp16 tensor or (hi, lo) pair;
    W: (hi, lo) pair of (N,K) fp16; bias (N) f32.  Returns, by mode:
      PM_HIDDEN    (Y_hi, Y_lo)                       relu, fp16 pair (M,N)
      PM_OUT_CM    out (B,N,points) f32, (Y_hi, Y_lo) relu
      PM_OUT_PM32  out (M,N) f32                      no activation
      PM_VOTE      vote_xyz (B,points,3), out (B,D,points) f32 L2-normalised, (Y_hi, Y_lo) (M,D)
      PM_LINEAR    (Y_hi, Y_lo)                       no activation, fp16 pair (M,N)"""
    X_hi, X_lo = X if isinstance(X, (tuple, list)) else (X, None)
    W_hi, W_lo = W
    _check(X_hi, "X_hi", HALF)
    _check(W_hi, "W_hi", HALF)
    _check(W_lo, "W_lo", HALF)
    _check(bias, "bias", torch.float32)
    _same_device(X_hi, W_hi, W_lo, bias)
    if X_lo is not None:
        _check(X_lo, "X_lo", HALF)
        assert X_lo.shape == X_hi.shape
    M, K = X_hi.shape
    N = W_hi.shape[0]
    assert W_hi.shape == (N, K) == W_lo.shape and bias.numel() == N and M % points_per_scene == 0
    B, dev = M // points_per_scene, X_hi.device
    Y_hi = Y_lo = out = vote_xyz = None
    D = N - 3 if mode == PM_VOTE else N
    if mode != PM_OUT_PM32:
        Y_hi = torch.empty((M, D), dtype=HALF, device=dev)
        Y_lo = torch.empty((M, D), dtype=HALF, device=dev) if want_lo else None
    if mode == PM_OUT_CM:
        out = torch.empty((B, N, points_per_scene), dtype=torch.float32, device=dev)
    elif mode == PM_OUT_PM32:
        out = torch.empty((M, N), dtype=torch.float32, device=dev)
    elif mode == PM_VOTE:
        _check(seed_cm, "seed_cm", torch.float32)
        _check(seed_xyz, "seed_xyz", torch.float32)
        assert seed_cm.shape == (B, D, points_per_scene) and seed_xyz.shape == (B, points_per_scene, 3)
        out = torch.empty((B, D, points_per_scene), dtype=torch.float32, device=dev)
        vote_xyz = torch.empty((B, points_per_scene, 3), dtype=torch.float32, device=dev)
    ptr = lambda t: t.data_ptr() if t is not None else None   # noqa: E731
    with torch.cuda.device(dev):
        _lib.call("spc_pm_linear", X_hi.data_ptr(), ptr(X_lo), M, K, W_hi.data_ptr(), W_lo.data_ptr(), bias.data_ptr(),
                  N, int(mode), int(points_per_scene), ptr(Y_hi), ptr(Y_lo), ptr(out), ptr(seed_cm), ptr(seed_xyz),
                  ptr(vote_xyz), int(_options.pm_n_tile), int(_options.pm_tiles_per_cta), _stream())
    if mode in (PM_HIDDEN, PM_LINEAR):
        return Y_hi, Y_lo
    if mode == PM_OUT_CM:
        return out, (Y_hi, Y_lo)
    if mode == PM_OUT_PM32:
        return out
    return vote_xyz, out, (Y_hi, Y_lo)


def _bn_workspace(C, device):
    nbytes = _lib.load().spc_bn_relu_workspace_bytes(int(C))
    return torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=device), nbytes


def _bn_sizes(y):
    """(B, C, S) of y (B,C,*); B may be 0 (a rank with an empty shard still takes part in the exchange)."""
    return y.shape[0], y.shape[1], math.prod(y.shape[2:])


def _per_channel(C, device):
    """Two per-channel f32 outputs: (save_mean, save_invstd) or (dgamma, dbeta)."""
    return (torch.empty(C, dtype=torch.float32, device=device), torch.empty(C, dtype=torch.float32, device=device))


def _pool_outputs(y):
    """(pooled, argmax, ymax, save_mean, save_invstd) of a max-pool forward of y (B,C,npoint,nsample)."""
    B, C, npoint, _ = y.shape
    pooled = torch.empty((B, C, npoint), dtype=y.dtype, device=y.device)
    argmax = torch.empty((B, C, npoint), dtype=torch.uint8, device=y.device)
    ymax = torch.empty((B, C, npoint), dtype=y.dtype, device=y.device)
    return (pooled, argmax, ymax) + _per_channel(C, y.device)


# The BatchNorm + ReLU wrappers below take y (and dz / dpool / ymax) as f32 or bf16 and return z / pooled / ymax / dy
# in the same dtype; gamma, beta, the saved statistics, dgamma / dbeta and the running statistics are f32.

def bn_relu_train_forward(y, gamma, beta, running_mean, running_var, momentum, eps):
    """Training-mode BatchNorm + ReLU of y (B,C,*) f32 or bf16 (pytorch_utils.py:11-36,39-64): returns
    (z, save_mean, save_invstd); running_mean / running_var (or None) are updated in place."""
    sfx = _storage(y, "y")
    _check(gamma, "gamma", torch.float32)
    _check(beta, "beta", torch.float32)
    _same_device(y, gamma, beta)
    B, C, S = _bn_sizes(y)
    z = torch.empty_like(y)
    mean, invstd = _per_channel(C, y.device)
    with torch.cuda.device(y.device):
        ws, nbytes = _bn_workspace(C, y.device)
        _lib.call("spc_bn_relu_train_forward" + sfx, y.data_ptr(), gamma.data_ptr(), beta.data_ptr(), B, C, S,
                  float(eps), float(momentum),
                  running_mean.data_ptr() if running_mean is not None else None,
                  running_var.data_ptr() if running_var is not None else None,
                  z.data_ptr(), mean.data_ptr(), invstd.data_ptr(), ws.data_ptr(), nbytes, _stream())
    return z, mean, invstd


def bn_relu_train_backward(dz, y, gamma, beta, mean, invstd):
    """-> (dy, dgamma, dbeta) for z = relu(batch_norm(y)) given dz."""
    sfx = _storage(y, "y")
    _check(dz, "dz", y.dtype)
    _same_device(dz, y)
    B, C, S = _bn_sizes(y)
    dy = torch.empty_like(y)
    dgamma, dbeta = _per_channel(C, y.device)
    with torch.cuda.device(y.device):
        ws, nbytes = _bn_workspace(C, y.device)
        _lib.call("spc_bn_relu_train_backward" + sfx, dz.data_ptr(), y.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                  mean.data_ptr(), invstd.data_ptr(), B, C, S, dy.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(),
                  ws.data_ptr(), nbytes, _stream())
    return dy, dgamma, dbeta


def bn_relu_maxpool_train_forward(y, gamma, beta, running_mean, running_var, momentum, eps):
    """y (B,C,npoint,nsample) f32 -> (pooled (B,C,npoint), argmax u8, ymax, save_mean, save_invstd):
    BatchNorm(train) + ReLU + max over nsample without materialising the activation
    (pytorch_utils.py:11-36 + pointnet2_modules.py:256-259).  Raises SpcUnsupported for nsample not in
    {16,32,64}."""
    sfx = _storage(y, "y")
    _same_device(y, gamma, beta)
    B, C, npoint, nsample = y.shape
    out = _pool_outputs(y)
    with torch.cuda.device(y.device):
        ws, nbytes = _bn_workspace(C, y.device)
        _lib.call("spc_bn_relu_maxpool_train_forward" + sfx, y.data_ptr(), gamma.data_ptr(), beta.data_ptr(), B, C,
                  npoint, nsample, float(eps), float(momentum),
                  running_mean.data_ptr() if running_mean is not None else None,
                  running_var.data_ptr() if running_var is not None else None,
                  *(t.data_ptr() for t in out), ws.data_ptr(), nbytes, _stream())
    return out


def bn_relu_maxpool_train_backward(dpool, argmax, ymax, y, gamma, beta, mean, invstd):
    """-> (dy (B,C,npoint,nsample), dgamma, dbeta)."""
    sfx = _storage(y, "y")
    _check(dpool, "dpool", y.dtype)
    _check(ymax, "ymax", y.dtype)
    _same_device(dpool, y)
    B, C, npoint, nsample = y.shape
    dy = torch.empty_like(y)
    dgamma, dbeta = _per_channel(C, y.device)
    with torch.cuda.device(y.device):
        _lib.call("spc_bn_relu_maxpool_train_backward" + sfx, dpool.data_ptr(), argmax.data_ptr(), ymax.data_ptr(),
                  y.data_ptr(), gamma.data_ptr(), beta.data_ptr(), mean.data_ptr(), invstd.data_ptr(), B, C,
                  npoint, nsample, dy.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), _stream())
    return dy, dgamma, dbeta


# ---- synchronised BatchNorm: the phases around the cross-rank exchange (include/spacap3d_ops.h) ----------------------
BN_SYNC_K = 3          # SPC_BN_SYNC_K: fp64 values per channel in an exchanged row


def _check_rows(rows, C, what):
    _check(rows, what, torch.float64)
    if rows.dim() < 2 or tuple(rows.shape[-2:]) != (C, BN_SYNC_K):
        raise RuntimeError("%s must have shape (..., %d, %d)" % (what, C, BN_SYNC_K))


def bn_relu_sync_stats(y, row):
    """This rank's per-channel (n, mean, M2) of y (B,C,*) f32 into row (C, BN_SYNC_K) f64; also the statistics phase
    of the max-pool variant."""
    sfx = _storage(y, "y")
    B, C, S = _bn_sizes(y)
    _check_rows(row, C, "row")
    _same_device(y, row)
    with torch.cuda.device(y.device):
        ws, nbytes = _bn_workspace(C, y.device)
        _lib.call("spc_bn_relu_sync_stats" + sfx, y.data_ptr(), B, C, S, row.data_ptr(), ws.data_ptr(), nbytes, _stream())


def bn_relu_sync_forward(y, gamma, beta, running_mean, running_var, momentum, eps, rows):
    """z = relu(batch_norm(y)) with the statistics combined from rows (world, C, BN_SYNC_K), every rank's
    bn_relu_sync_stats row: returns (z, save_mean, save_invstd); running_mean / running_var (or None) are updated
    in place with the global mean and unbiased variance."""
    sfx = _storage(y, "y")
    _check(gamma, "gamma", torch.float32)
    _check(beta, "beta", torch.float32)
    B, C, S = _bn_sizes(y)
    _check_rows(rows, C, "rows")
    _same_device(y, gamma, beta, rows)
    z = torch.empty_like(y)
    mean, invstd = _per_channel(C, y.device)
    with torch.cuda.device(y.device):
        _lib.call("spc_bn_relu_sync_forward" + sfx, y.data_ptr(), gamma.data_ptr(), beta.data_ptr(), B, C, S,
                  rows.shape[0], rows.data_ptr(), float(eps), float(momentum),
                  running_mean.data_ptr() if running_mean is not None else None,
                  running_var.data_ptr() if running_var is not None else None,
                  z.data_ptr(), mean.data_ptr(), invstd.data_ptr(), _stream())
    return z, mean, invstd


def bn_relu_sync_backward_reduce(dz, y, gamma, beta, mean, invstd, row):
    """-> (dgamma, dbeta) of this rank; writes its (n, sum dm, sum dm * xhat) into row (C, BN_SYNC_K) f64."""
    sfx = _storage(y, "y")
    _check(dz, "dz", y.dtype)
    B, C, S = _bn_sizes(y)
    _check_rows(row, C, "row")
    _same_device(dz, y, row)
    dgamma, dbeta = _per_channel(C, y.device)
    with torch.cuda.device(y.device):
        ws, nbytes = _bn_workspace(C, y.device)
        _lib.call("spc_bn_relu_sync_backward_reduce" + sfx, dz.data_ptr(), y.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                  mean.data_ptr(), invstd.data_ptr(), B, C, S, dgamma.data_ptr(), dbeta.data_ptr(), row.data_ptr(),
                  ws.data_ptr(), nbytes, _stream())
    return dgamma, dbeta


def bn_relu_sync_backward(dz, y, gamma, beta, mean, invstd, rows):
    """-> dy from dz, y and every rank's bn_relu_sync_backward_reduce row (rows (world, C, BN_SYNC_K))."""
    sfx = _storage(y, "y")
    _check(dz, "dz", y.dtype)
    B, C, S = _bn_sizes(y)
    _check_rows(rows, C, "rows")
    _same_device(dz, y, rows)
    dy = torch.empty_like(y)
    with torch.cuda.device(y.device):
        ws, nbytes = _bn_workspace(C, y.device)
        _lib.call("spc_bn_relu_sync_backward" + sfx, dz.data_ptr(), y.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                  mean.data_ptr(), invstd.data_ptr(), B, C, S, rows.shape[0], rows.data_ptr(), dy.data_ptr(),
                  ws.data_ptr(), nbytes, _stream())
    return dy


def bn_relu_maxpool_sync_forward(y, gamma, beta, running_mean, running_var, momentum, eps, rows):
    """bn_relu_maxpool_train_forward with the statistics combined from rows (world, C, BN_SYNC_K), every rank's
    bn_relu_sync_stats row of its y (B,C,npoint,nsample): -> (pooled, argmax, ymax, save_mean, save_invstd)."""
    sfx = _storage(y, "y")
    _check(gamma, "gamma", torch.float32)
    _check(beta, "beta", torch.float32)
    B, C, npoint, nsample = y.shape
    _check_rows(rows, C, "rows")
    _same_device(y, gamma, beta, rows)
    out = _pool_outputs(y)
    with torch.cuda.device(y.device):
        _lib.call("spc_bn_relu_maxpool_sync_forward" + sfx, y.data_ptr(), gamma.data_ptr(), beta.data_ptr(), B, C,
                  npoint, nsample, rows.shape[0], rows.data_ptr(), float(eps), float(momentum),
                  running_mean.data_ptr() if running_mean is not None else None,
                  running_var.data_ptr() if running_var is not None else None,
                  *(t.data_ptr() for t in out), _stream())
    return out


def bn_relu_maxpool_sync_backward_reduce(dpool, ymax, y, gamma, beta, mean, invstd, row):
    """-> (dgamma, dbeta) of this rank for the max-pool variant; writes its row (C, BN_SYNC_K) f64."""
    sfx = _storage(dpool, "dpool")
    _check(ymax, "ymax", dpool.dtype)
    _same_device(dpool, ymax, row)
    B, C, npoint, nsample = y.shape
    _check_rows(row, C, "row")
    dgamma, dbeta = _per_channel(C, dpool.device)
    with torch.cuda.device(dpool.device):
        _lib.call("spc_bn_relu_maxpool_sync_backward_reduce" + sfx, dpool.data_ptr(), ymax.data_ptr(), gamma.data_ptr(),
                  beta.data_ptr(), mean.data_ptr(), invstd.data_ptr(), B, C, npoint, nsample, dgamma.data_ptr(),
                  dbeta.data_ptr(), row.data_ptr(), _stream())
    return dgamma, dbeta


def bn_relu_maxpool_sync_backward(dpool, argmax, ymax, y, gamma, beta, mean, invstd, rows):
    """-> dy (B,C,npoint,nsample) from dpool and every rank's bn_relu_maxpool_sync_backward_reduce row."""
    sfx = _storage(y, "y")
    _check(dpool, "dpool", y.dtype)
    B, C, npoint, nsample = y.shape
    _check_rows(rows, C, "rows")
    _same_device(dpool, y, rows)
    dy = torch.empty_like(y)
    with torch.cuda.device(y.device):
        ws, nbytes = _bn_workspace(C, y.device)
        _lib.call("spc_bn_relu_maxpool_sync_backward" + sfx, dpool.data_ptr(), argmax.data_ptr(), ymax.data_ptr(),
                  y.data_ptr(), gamma.data_ptr(), beta.data_ptr(), mean.data_ptr(), invstd.data_ptr(), B, C,
                  npoint, nsample, rows.shape[0], rows.data_ptr(), dy.data_ptr(), ws.data_ptr(), nbytes, _stream())
    return dy


def box_point_counts(points, corners):
    """points (B,N,>=3) f32, corners (B,K,8,3) f64 -> (B,K) int32 points inside each box
    (ap_helper.py:69-79: extract_pc_in_box3d per predicted box)."""
    _check(points, "points", torch.float32)
    _check(corners, "corners", torch.float64)
    _same_device(points, corners)
    B, N, stride = points.shape
    K = corners.shape[1]
    counts = torch.empty((B, K), dtype=torch.int32, device=points.device)
    with torch.cuda.device(points.device):
        _lib.call("spc_box_point_counts", points.data_ptr(), int(stride), corners.data_ptr(), B, N, K,
                  counts.data_ptr(), _stream())
    return counts


def nms_boxes(corners, score, cls=None, valid=None, mode=2, old_type=False, iou_threshold=0.25):
    """corners (B,K,8,3) f64, score (B,K) f32, cls (B,K) i64, valid (B,K) i32 -> pick (B,K) int32.
    mode 0/1/2 = nms_2d_faster / nms_3d_faster / nms_3d_faster_samecls (utils/nms.py:39-147)."""
    _check(corners, "corners", torch.float64)
    _check(score, "score", torch.float32)
    if cls is not None:
        _check(cls, "cls", torch.int64)
    if valid is not None:
        _check(valid, "valid", torch.int32)
    _same_device(corners, score)
    B, K = score.shape
    pick = torch.empty((B, K), dtype=torch.int32, device=score.device)
    with torch.cuda.device(score.device):
        _lib.call("spc_nms_boxes", corners.data_ptr(), score.data_ptr(),
                  cls.data_ptr() if cls is not None else None, valid.data_ptr() if valid is not None else None,
                  B, K, int(mode), int(bool(old_type)), float(iou_threshold), pick.data_ptr(), _stream())
    return pick


# ---- input pipeline (SURVEY row N4; lib/dataset.py:291-531) ------------------------------------------------------

def scene_floor_height(verts, col=2, quantile=None):
    """verts (M,stride) f32 -> (1,) f32 = np.percentile(verts[:, col], 0.99) (lib/dataset.py:331)."""
    import numpy as np
    _check(verts, "verts", torch.float32)
    _same_device(verts)
    M, stride = verts.shape
    if quantile is None:
        quantile = float(np.float32(0.99) / np.float32(100))        # numpy's float32 quantile for a float32 column
    out = torch.empty(1, dtype=torch.float32, device=verts.device)
    with torch.cuda.device(verts.device):
        _lib.call("spc_scene_floor_height", verts.data_ptr(), int(M), int(stride), int(col), float(quantile),
                  out.data_ptr(), _stream())
    return out


def prepare_point_clouds(verts, row0, choices, multiview=None, floor_height=None, aug=None, mean_rgb=None,
                         use_color=False, use_normal=False):
    """Packed vertex table (rows,stride) f32 + row0 (B,) i64 + choices (B,P) i32 -> point_clouds (B,P,C) f32
    (lib/dataset.py:309-335 and the augmentation of :366-404; `aug` (B,32) f64, see include/spacap3d_ops.h)."""
    _check(verts, "verts", torch.float32)
    _check(row0, "row0", torch.int64)
    _check(choices, "choices", torch.int32)
    others = [row0, choices]
    n_mv = 0
    if multiview is not None:
        _check(multiview, "multiview", torch.float32)
        n_mv = multiview.shape[1]
        others.append(multiview)
    if floor_height is not None:
        _check(floor_height, "floor_height", torch.float32)
        others.append(floor_height)
    if aug is not None:
        _check(aug, "aug", torch.float64)
        if tuple(aug.shape) != (choices.shape[0], 32):
            raise RuntimeError("aug must be (B,32)")
        others.append(aug)
    _same_device(verts, *others)
    B, P = choices.shape
    if use_color and mean_rgb is None:
        raise RuntimeError("use_color needs mean_rgb")
    mr = [float(v) for v in (mean_rgb if mean_rgb is not None else (0.0, 0.0, 0.0))]
    C = 3 + (3 if use_color else 0) + (3 if use_normal else 0) + n_mv + (1 if floor_height is not None else 0)
    out = torch.empty((B, P, C), dtype=torch.float32, device=verts.device)
    with torch.cuda.device(verts.device):
        _lib.call("spc_prepare_point_clouds", verts.data_ptr(), int(verts.shape[1]),
                  multiview.data_ptr() if multiview is not None else None, int(n_mv), row0.data_ptr(),
                  choices.data_ptr(), floor_height.data_ptr() if floor_height is not None else None,
                  aug.data_ptr() if aug is not None else None, mr[0], mr[1], mr[2], B, P, int(bool(use_color)),
                  int(bool(use_normal)), out.data_ptr(), _stream())
    return out


def vote_labels(point_clouds, instance_labels, semantic_labels, row0, choices, max_instances, sem_mask):
    """-> vote_label (B,P,9) f32, vote_label_mask (B,P) i64, overflow (1,) i32   (lib/dataset.py:421-431)."""
    _check(point_clouds, "point_clouds", torch.float32)
    _check(instance_labels, "instance_labels", torch.int32)
    _check(semantic_labels, "semantic_labels", torch.int32)
    _check(row0, "row0", torch.int64)
    _check(choices, "choices", torch.int32)
    _same_device(point_clouds, instance_labels, semantic_labels, row0, choices)
    B, P, C = point_clouds.shape
    dev = point_clouds.device
    votes = torch.empty((B, P, 9), dtype=torch.float32, device=dev)
    mask = torch.empty((B, P), dtype=torch.int64, device=dev)
    overflow = torch.empty(1, dtype=torch.int32, device=dev)
    nbytes = _lib.load().spc_vote_labels_workspace_bytes(B, int(max_instances))
    ws = torch.empty(max(1, nbytes // 4), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.call("spc_vote_labels", point_clouds.data_ptr(), int(C), instance_labels.data_ptr(),
                  semantic_labels.data_ptr(), row0.data_ptr(), choices.data_ptr(), B, P, int(max_instances),
                  int(sem_mask), votes.data_ptr(), mask.data_ptr(), overflow.data_ptr(), ws.data_ptr(), nbytes,
                  _stream())
    return votes, mask, overflow


def augment_boxes(boxes, aug):
    """boxes (B,K,6) f64 + aug (B,32) f64 -> (B,K,6) f64   (lib/dataset.py:369-404)."""
    _check(boxes, "boxes", torch.float64)
    _check(aug, "aug", torch.float64)
    _same_device(boxes, aug)
    B, K, _ = boxes.shape
    out = torch.empty_like(boxes)
    with torch.cuda.device(boxes.device):
        _lib.call("spc_augment_boxes", boxes.data_ptr(), aug.data_ptr(), B, K, out.data_ptr(), _stream())
    return out
