"""Same public API as the reference's lib/pointnet2/pointnet2_modules.py: the set-abstraction
and feature-propagation layers SpaCap3D's detector is built from
(PointnetSAModuleVotes :165-276, PointnetFPModule :361-421; plus _PointnetSAModuleBase,
PointnetSAModuleMSG, PointnetSAModule, PointnetSAModuleMSGVotes, PointnetLFPModuleMSG for API
completeness).  Parameter trees (`mlp_module.layer{i}.conv/.bn.bn`, `mlp.layer{i}...`) are the
reference's, so its checkpoints load unchanged (SURVEY F11).

All point-set work runs on this package's sm_100a kernels via pointnet2_utils.
"""
from typing import List

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import pointnet2_utils
from . import pytorch_utils as pt_utils
from . import _ext
from . import _lib

# When False every module runs the reference's exact op sequence (FPS -> gather -> ball query ->
# 2x grouping -> cat -> MLP -> pool) through `_ext`; used by the parity tests and by
# bench.py --impl reference, which swaps `_ext` for the reference's own extension.
FAST_PATHS = True


def _sample_centres(xyz, npoint, inds=None):
    """FPS (unless indices are supplied) + gather of the sampled coordinates.
    Returns (new_xyz (B,npoint,3) or None, inds)."""
    if npoint is None:
        return None, inds
    needs_grad = torch.is_grad_enabled() and xyz.requires_grad
    if inds is None and not needs_grad and FAST_PATHS:
        # one kernel: the FPS epilogue already holds the winners' coordinates.  Centres produced by
        # an FPS are tagged so that the next layer can try the verified "already FPS-ordered"
        # shortcut (exact: see spc_furthest_point_sampling_ex).
        # `_spc_fps_strict` carries the producing call's per-scene "strict sequence" flags (tracked exactly by the
        # bucketed sampler, implied by a successful proof): flagged scenes need neither the proof nor the rounds.
        hint = bool(getattr(xyz, "_spc_fps_ordered", False))
        known = getattr(xyz, "_spc_fps_strict", None) if hint and npoint <= xyz.shape[1] else None
        inds, new_xyz, strict = _ext.furthest_point_sampling_with_xyz(
            xyz.contiguous(), npoint, hint_ordered=hint, known_ordered=known, want_strict=True)
        new_xyz._spc_fps_ordered = True
        new_xyz._spc_fps_strict = strict
        return new_xyz, inds
    if inds is None:
        inds = pointnet2_utils.furthest_point_sample(xyz, npoint)
    xyz_flipped = xyz.transpose(1, 2).contiguous()
    new_xyz = pointnet2_utils.gather_operation(xyz_flipped, inds).transpose(1, 2).contiguous()
    return new_xyz, inds


INLINE_MAX_FEATURES = 13   # raw feature channels the fused kernel evaluates in-line (layer 0)
PAD_TRAINING_CHANNELS = True   # training: pad 3+C grouped channels to a multiple of 4 (aligned conv GEMMs; 8 in bf16)


def _autocast_bf16():
    """torch.bfloat16 when the convolutions that follow will run in bf16 under CUDA autocast, else None."""
    if torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == torch.bfloat16:
        return torch.bfloat16
    return None


def attach_pm(t, pm, pm_lo=None):
    """Tag fp32 tensor `t` (B,C,n) with its point-major 16-bit copy `pm` (B,n,C) for the next fast-path stage
    (optionally as a hi + lo fp16 pair, t ~= pm + pm_lo to fp32 accuracy).
    The tag records t's version counter and storage pointer: any in-place edit of `t` between layers
    (`features.mul_(mask)`, in-place dropout, `copy_`) invalidates the copy instead of being silently ignored."""
    t._spc_pm = (pm, t._version, t.data_ptr(), pm_lo)
    return t


def get_pm_pair(t):
    """(hi, lo-or-None) attached to `t` by attach_pm, or (None, None) when absent, stale or mis-shaped."""
    tag = getattr(t, "_spc_pm", None)
    if tag is None:
        return None, None
    pm, version, ptr, pm_lo = tag
    if version != t._version or ptr != t.data_ptr() or pm.device != t.device or t.dim() != 3 \
            or pm.shape[:2] != (t.shape[0], t.shape[2]) or not t.shape[1] <= pm.shape[2] < t.shape[1] + 8:
        return None, None     # (the channel dimension of the copy may be zero-padded to a multiple of 8)
    return pm, pm_lo


def get_pm(t):
    """The point-major copy attached to `t` by attach_pm, or None when absent, stale or mis-shaped."""
    return get_pm_pair(t)[0]


# BN-folded weight caches live OUTSIDE the modules' __dict__: nn.DataParallel's replicate() shallow-copies that
# dict, which would make every replica (one per device and thread) share and overwrite one cache object.
# Keyed weakly by module, so a replica's cache dies with the replica.
import threading as _threading
import warnings
import weakref as _weakref
_WARNED_UNFUSED = _weakref.WeakSet()
_CACHES = _weakref.WeakKeyDictionary()
_CACHES_LOCK = _threading.Lock()


def _cache_of(module, factory):
    with _CACHES_LOCK:
        c = _CACHES.get(module)
        if c is None:
            c = _CACHES[module] = factory()
        return c


def invalidate_folded_caches(model=None):
    """Drop the cached BN-folded weights of `model`'s modules (all modules when None).  The caches refresh
    themselves when a parameter / running statistic changes through autograd-visible in-place ops (tensor version
    counters); writes through `param.data` or raw pointers do not bump a version and need this call."""
    with _CACHES_LOCK:
        if model is None:
            _CACHES.clear()
        else:
            for m in model.modules():
                _CACHES.pop(m, None)


def _fold_conv_bn(block):
    """(W (Cout,Cin) f32, b (Cout) f32) of one SharedMLP block with eval-mode BN folded in, or
    None when the block is not conv[+bn]+ReLU."""
    conv = getattr(block, "conv", None)
    act = getattr(block, "activation", None)
    if conv is None or not isinstance(act, nn.ReLU) or conv.kernel_size != (1, 1):
        return None
    W = conv.weight.detach().reshape(conv.out_channels, conv.in_channels).float()
    norm = getattr(block, "bn", None)
    if norm is not None:
        bn = norm.bn
        if bn.running_mean is None:
            return None
        scale = bn.weight.detach() / torch.sqrt(bn.running_var + bn.eps)
        shift = bn.bias.detach() - bn.running_mean * scale
        if conv.bias is not None:
            shift = shift + conv.bias.detach() * scale
        return W * scale[:, None], shift.float()
    b = conv.bias.detach().float() if conv.bias is not None else torch.zeros(conv.out_channels, device=W.device)
    return W, b


class _FoldedMLP:
    """Cache of the BN-folded weights of a 3-layer SharedMLP (refreshed when any parameter or
    running statistic changes, tracked through tensor versions)."""

    def __init__(self):
        self.key = None
        self.data = None
        self._w0f_t = None
        self._w0x = None

    def w0f(self, W0):
        """((C1, Cf) fp16 hi, lo): feature columns of the folded conv0 for the projection layer (spc_pm_linear),
        plus a zero bias."""
        if self._w0f_t is None:
            self._w0f_t = (_ext.split_half(W0[:, 3:].contiguous()),
                           torch.zeros(W0.shape[0], dtype=torch.float32, device=W0.device))
        return self._w0f_t

    def w0x(self, W0):
        """(C1, 3) f32: xyz columns of the folded conv0."""
        if self._w0x is None:
            self._w0x = W0[:, :3].contiguous()
        return self._w0x

    def get(self, mlp):
        tensors = [t for t in list(mlp.parameters()) + list(mlp.buffers())]
        key = tuple((t.data_ptr(), t._version, t.device) for t in tensors)
        if key != self.key:
            self.key = key
            self.data = None
            self._w0f_t = self._w0x = None
            blocks = list(mlp.children())
            if len(blocks) == 3:
                folded = [_fold_conv_bn(b) for b in blocks]
                if all(f is not None for f in folded):
                    (W0, b0), (W1, b1), (W2, b2) = folded
                    self.data = (W0.contiguous(), b0.contiguous(),
                                 W1.to(_ext.HALF).contiguous(), b1.contiguous(),
                                 W2.to(_ext.HALF).contiguous(), b2.contiguous())
        return self.data


def fold_conv_bn_pair(conv, bn):
    """(W (Cout,Cin) f32, b (Cout) f32) of a 1x1 conv followed by an optional eval-mode BatchNorm."""
    W = conv.weight.detach().reshape(conv.out_channels, conv.in_channels).float()
    b = conv.bias.detach().float() if conv.bias is not None else torch.zeros(conv.out_channels, device=W.device)
    if bn is not None:
        scale = bn.weight.detach() / torch.sqrt(bn.running_var + bn.eps)
        W = W * scale[:, None]
        b = (b - bn.running_mean) * scale + bn.bias.detach()
    return W, b


class FoldedChain:
    """Cache of a conv(+BN)(+ReLU) chain as operands of spc_pm_linear: [((W_hi, W_lo) (Cout,Cin) fp16 pair, b f32)],
    refreshed when a parameter / running statistic changes (tensor versions)."""

    def __init__(self):
        self.key = None
        self.layers = None

    def get(self, pairs, last_rows_rotate=0):
        """pairs: list of (conv, bn_or_None).  last_rows_rotate = r moves the first r output channels of the LAST
        layer behind the others (the voting tail wants conv3's feature rows first, its xyz-offset rows last)."""
        tensors = []
        for conv, bn in pairs:
            tensors += list(conv.parameters()) + (list(bn.parameters()) + list(bn.buffers()) if bn is not None else [])
        key = tuple((t.data_ptr(), t._version, t.device) for t in tensors)
        if key != self.key:
            self.key = key
            self.layers = []
            for conv, bn in pairs:
                W, b = fold_conv_bn_pair(conv, bn)
                if last_rows_rotate and conv is pairs[-1][0]:
                    r = last_rows_rotate
                    W, b = torch.cat([W[r:], W[:r]], 0), torch.cat([b[r:], b[:r]], 0)
                self.layers.append((_ext.split_half(W.contiguous()), b.contiguous()))
        return self.layers


def fast_eval_ok(*tensors):
    """The fp16 point-major fast paths apply in eval-style use only: no autograd, CUDA tensors."""
    return FAST_PATHS and not torch.is_grad_enabled() and all(t is not None and t.is_cuda for t in tensors)


def _pool_max(x):
    """(B,C,npoint,nsample) -> (B,C,npoint)"""
    return F.max_pool2d(x, kernel_size=[1, x.size(3)]).squeeze(-1)


def _build_groupers(npoint, radii, nsamples, mlps, bn, use_xyz, sample_uniformly):
    groupers, nets = nn.ModuleList(), nn.ModuleList()
    for radius, nsample, mlp_spec in zip(radii, nsamples, mlps):
        groupers.append(
            pointnet2_utils.QueryAndGroup(radius, nsample, use_xyz=use_xyz,
                                          sample_uniformly=sample_uniformly)
            if npoint is not None else pointnet2_utils.GroupAll(use_xyz))
        if use_xyz:
            mlp_spec[0] += 3          # mutates the caller's list, like the reference (:207-209)
        nets.append(pt_utils.SharedMLP(mlp_spec, bn=bn))
    return groupers, nets


class _PointnetSAModuleBase(nn.Module):
    def __init__(self):
        super().__init__()
        self.npoint = None
        self.groupers = None
        self.mlps = None

    def forward(self, xyz: torch.Tensor, features: torch.Tensor = None):
        """xyz (B,N,3), features (B,C,N) -> new_xyz (B,npoint,3), new_features (B,sum C_k,npoint)"""
        new_xyz, _ = _sample_centres(xyz, self.npoint)
        outs = [_pool_max(mlp(grouper(xyz, new_xyz, features)))
                for grouper, mlp in zip(self.groupers, self.mlps)]
        return new_xyz, torch.cat(outs, dim=1)


class PointnetSAModuleMSG(_PointnetSAModuleBase):
    """Set abstraction with multi-scale grouping."""

    def __init__(self, *, npoint: int, radii: List[float], nsamples: List[int],
                 mlps: List[List[int]], bn: bool = True, use_xyz: bool = True,
                 sample_uniformly: bool = False):
        super().__init__()
        assert len(radii) == len(nsamples) == len(mlps)
        self.npoint = npoint
        self.groupers, self.mlps = _build_groupers(npoint, radii, nsamples, mlps, bn, use_xyz,
                                                   sample_uniformly)


class PointnetSAModule(PointnetSAModuleMSG):
    """Single-scale set abstraction."""

    def __init__(self, *, mlp: List[int], npoint: int = None, radius: float = None,
                 nsample: int = None, bn: bool = True, use_xyz: bool = True):
        super().__init__(mlps=[mlp], npoint=npoint, radii=[radius], nsamples=[nsample], bn=bn,
                         use_xyz=use_xyz)


class PointnetSAModuleVotes(nn.Module):
    """Set abstraction that also returns the sampled indices (VoteNet needs them for vote
    supervision).  forward(xyz, features=None, inds=None) -> (new_xyz, new_features, inds)."""

    def __init__(self, *, mlp: List[int], npoint: int = None, radius: float = None,
                 nsample: int = None, bn: bool = True, use_xyz: bool = True,
                 pooling: str = 'max', sigma: float = None, normalize_xyz: bool = False,
                 sample_uniformly: bool = False, ret_unique_cnt: bool = False):
        super().__init__()
        self.npoint = npoint
        self.radius = radius
        self.nsample = nsample
        self.pooling = pooling
        self.use_xyz = use_xyz
        self.sigma = sigma if sigma is not None else (self.radius / 2 if self.radius is not None else None)
        self.normalize_xyz = normalize_xyz
        self.ret_unique_cnt = ret_unique_cnt
        if npoint is not None:
            self.grouper = pointnet2_utils.QueryAndGroup(
                radius, nsample, use_xyz=use_xyz, ret_grouped_xyz=True,
                normalize_xyz=normalize_xyz, sample_uniformly=sample_uniformly,
                ret_unique_cnt=ret_unique_cnt)
        else:
            self.grouper = pointnet2_utils.GroupAll(use_xyz, ret_grouped_xyz=True)
        mlp_spec = mlp
        if use_xyz and len(mlp_spec) > 0:
            mlp_spec[0] += 3
        self.mlp_module = pt_utils.SharedMLP(mlp_spec, bn=bn)

    def forward(self, xyz: torch.Tensor, features: torch.Tensor = None, inds: torch.Tensor = None):
        """xyz (B,N,3), features (B,C,N), inds (B,npoint) optional ->
        new_xyz (B,npoint,3), new_features (B,mlp[-1],npoint), inds (B,npoint) int32"""
        if inds is not None:
            assert inds.shape[1] == self.npoint
        new_xyz, inds = _sample_centres(xyz, self.npoint, inds)
        fused = self._forward_fused(xyz, new_xyz, features)
        if fused is not None:
            return new_xyz, fused, inds
        if features is not None and not features.is_contiguous():
            features = features.contiguous()      # (a caller may hand in a channel-major VIEW of a point-major cloud)
        # training on the GPU: zero-pad the grouped tensor to a multiple of 4 channels (aligned GEMM rows, see
        # QueryAndGroup.forward); the first SharedMLP block pads its weight to match -- same values either way.
        # Under bf16 autocast the grouped tensor is built in bf16 (the conv's input dtype) and padded to a multiple
        # of 8 channels, 16-byte rows of bf16.
        train_gpu = (self.training and xyz.is_cuda and features is not None and len(self.mlp_module) > 0
                     and isinstance(self.grouper, pointnet2_utils.QueryAndGroup))
        group_kw = {}
        amp = _autocast_bf16() if train_gpu else None
        if amp is not None:
            group_kw["dtype"] = amp
        if train_gpu and PAD_TRAINING_CHANNELS:
            group_kw["pad_channels_to"] = 8 if amp is not None else 4
        grouped_features, grouped_xyz = self.grouper(xyz, new_xyz, features, **group_kw)
        if (self.pooling == 'max' and self.training and grouped_features.is_cuda and len(self.mlp_module) > 0
                and pt_utils.FUSED_BN_RELU_TRAINING):
            # training: the last block's BatchNorm + ReLU + max-pool run as one kernel pair (csrc/bn_relu.cu)
            return new_xyz, self.mlp_module.forward_max_pooled(grouped_features), inds
        new_features = self.mlp_module(grouped_features)      # (B, mlp[-1], npoint, nsample)
        if self.pooling == 'max':
            new_features = F.max_pool2d(new_features, kernel_size=[1, new_features.size(3)])
        elif self.pooling == 'avg':
            new_features = F.avg_pool2d(new_features, kernel_size=[1, new_features.size(3)])
        elif self.pooling == 'rbf':
            # radial-basis weighting of the neighbours, normalised by nsample
            rbf = torch.exp(-1 * grouped_xyz.pow(2).sum(1, keepdim=False) / (self.sigma ** 2) / 2)
            new_features = torch.sum(new_features * rbf.unsqueeze(1), -1, keepdim=True) / float(self.nsample)
        new_features = new_features.squeeze(-1)
        return new_xyz, new_features, inds


    # -- fused eval path ---------------------------------------------------------------------------
    def _forward_fused(self, xyz, new_xyz, features):
        """ball query -> ONE kernel (gather, relative xyz, 3 x [1x1 conv + folded BN + ReLU] with
        the wide convs on tcgen05, max-pool).  Eval mode without autograd only; returns None when
        not applicable so that the caller runs the reference op sequence on the unfused kernels."""
        if (not FAST_PATHS or self.training or torch.is_grad_enabled() or self.npoint is None
                or self.pooling != 'max' or not self.use_xyz or not xyz.is_cuda
                or not isinstance(self.grouper, pointnet2_utils.QueryAndGroup)
                or self.grouper.sample_uniformly or (features is not None and features.dtype != torch.float32)):
            return None
        cache = _cache_of(self, _FoldedMLP)
        folded = cache.get(self.mlp_module)
        if folded is None:
            return None
        W0, b0, W1, b1, W2, b2 = folded
        Cf = 0 if features is None else features.shape[1]
        if W0.shape[1] != 3 + Cf:
            return None
        radius = float(self.radius) if self.normalize_xyz else 1.0
        xyz = xyz.contiguous()
        idx = pointnet2_utils.ball_query(self.radius, self.nsample, xyz, new_xyz)
        try:
            if Cf <= INLINE_MAX_FEATURES:
                feat = None if features is None else features.contiguous()
                out, out_pm = _ext.sa_fused_forward(xyz, new_xyz, idx, W0, b0, W1, b1, W2, b2, feat=feat,
                                                    radius=radius, want_point_major=True)
            else:
                # conv0 hoisted out of the grouping: ONE tcgen05 layer over the n points gives the
                # per-point feature projection; the xyz columns stay in fp32 inside the kernel
                pm, pm_lo = get_pm_pair(features)              # point-major fp16 copy from the producer
                if pm is None:
                    pm, pm_lo = _ext.split_half(features.transpose(1, 2))
                Wp, zero = cache.w0f(W0)
                Kp = pm.shape[2]                               # Cf, or Cf padded to a multiple of 8 by the producer
                if Kp % 8:                                     # TMA rows must be 16-byte multiples: pad with zeros
                    Kp = (Cf + 7) // 8 * 8
                    pm = torch.nn.functional.pad(pm, (0, Kp - Cf))
                    pm_lo = torch.nn.functional.pad(pm_lo, (0, Kp - Cf)) if pm_lo is not None else None
                if Wp[0].shape[1] != Kp:
                    Wp = tuple(torch.nn.functional.pad(t, (0, Kp - t.shape[1])) for t in Wp)
                    cache._w0f_t = (Wp, zero)
                Bn = pm.shape[0] * pm.shape[1]
                X = pm.reshape(Bn, Kp) if pm_lo is None else (pm.reshape(Bn, Kp), pm_lo.reshape(Bn, Kp))
                G, _ = _ext.pm_linear(X, Wp, zero, _ext.PM_LINEAR, pm.shape[1], want_lo=False)
                G = G.view(pm.shape[0], pm.shape[1], -1)
                out, out_pm = _ext.sa_fused_forward(xyz, new_xyz, idx, cache.w0x(W0), b0, W1, b1, W2, b2,
                                                    G=G, radius=radius, want_point_major=True)
            return attach_pm(out, out_pm)       # lets the next layer skip its transpose + cast
        except _lib.SpcUnsupported as e:
            # not an error -- the unfused kernels give the same result -- but never silent: a configuration that
            # falls off the fused path is 10-20x slower in this layer
            if self not in _WARNED_UNFUSED:
                _WARNED_UNFUSED.add(self)
                warnings.warn("PointnetSAModuleVotes: no fused set-abstraction kernel for this layer (%s); using the "
                              "unfused kernels" % e, RuntimeWarning, stacklevel=3)
            return None


class PointnetSAModuleMSGVotes(nn.Module):
    """Multi-scale set abstraction returning the sampled indices."""

    def __init__(self, *, mlps: List[List[int]], npoint: int, radii: List[float],
                 nsamples: List[int], bn: bool = True, use_xyz: bool = True,
                 sample_uniformly: bool = False):
        super().__init__()
        assert len(mlps) == len(nsamples) == len(radii)
        self.npoint = npoint
        self.groupers, self.mlps = _build_groupers(npoint, radii, nsamples, mlps, bn, use_xyz,
                                                   sample_uniformly)

    def forward(self, xyz: torch.Tensor, features: torch.Tensor = None, inds: torch.Tensor = None):
        new_xyz, inds = _sample_centres(xyz, self.npoint, inds)
        outs = [_pool_max(mlp(grouper(xyz, new_xyz, features)))
                for grouper, mlp in zip(self.groupers, self.mlps)]
        return new_xyz, torch.cat(outs, dim=1), inds


class PointnetFPModule(nn.Module):
    """Feature propagation: inverse-distance 3-NN interpolation + skip concat + SharedMLP."""

    def __init__(self, *, mlp: List[int], bn: bool = True):
        super().__init__()
        self.mlp = pt_utils.SharedMLP(mlp, bn=bn)

    def forward(self, unknown: torch.Tensor, known: torch.Tensor, unknow_feats: torch.Tensor,
                known_feats: torch.Tensor) -> torch.Tensor:
        """unknown (B,n,3), known (B,m,3), unknow_feats (B,C1,n), known_feats (B,C2,m)
        -> (B,mlp[-1],n)"""
        fast = self._forward_fast(unknown, known, unknow_feats, known_feats)
        if fast is not None:
            return fast
        if known is not None:
            dist, idx = pointnet2_utils.three_nn(unknown, known)
            dist_recip = 1.0 / (dist + 1e-8)
            norm = torch.sum(dist_recip, dim=2, keepdim=True)
            weight = dist_recip / norm
            interpolated_feats = pointnet2_utils.three_interpolate(known_feats, idx, weight)
        else:
            interpolated_feats = known_feats.expand(*known_feats.size()[0:2], unknown.size(1))
        new_features = interpolated_feats if unknow_feats is None else \
            torch.cat([interpolated_feats, unknow_feats], dim=1)
        return self.mlp(new_features.unsqueeze(-1)).squeeze(-1)


    # -- fp16 point-major eval path -------------------------------------------------------------------
    def _forward_fast(self, unknown, known, unknow_feats, known_feats):
        """three_nn+weights (1 kernel) -> interpolate+concat (1 kernel, point-major fp16) -> one tcgen05 launch per
        MLP layer (spc_pm_linear: fp16-pair operands, fp32-grade; the last one also writes the API's channel-major
        fp32 tensor).  Needs the point-major copies that the fused SA / FP kernels attach to their outputs."""
        if self.training or known is None or not fast_eval_ok(unknown, known, unknow_feats, known_feats):
            return None
        kpm, spm = get_pm(known_feats), get_pm(unknow_feats)
        if kpm is None or spm is None or known.shape[1] < 3 or kpm.shape[2] % 8 or spm.shape[2] % 8:
            return None
        pairs = []
        for block in self.mlp.children():
            conv, norm, act = getattr(block, "conv", None), getattr(block, "bn", None), getattr(block, "activation", None)
            if conv is None or not isinstance(act, nn.ReLU) or conv.kernel_size != (1, 1):
                return None
            pairs.append((conv, norm.bn if norm is not None else None))
        chain = _cache_of(self, FoldedChain).get(pairs)
        if chain[0][0][0].shape[1] != kpm.shape[2] + spm.shape[2] or any(W[0].shape[1] % 64 or W[0].shape[0] % 32
                                                                         for W, _ in chain):
            return None
        idx, weight = _ext.three_nn_weights(unknown.contiguous(), known.contiguous())
        X = _ext.interp_cat_pm(kpm, idx, weight, spm)
        B, n = X.shape[0], X.shape[1]
        h = X.view(B * n, -1)
        for W, b in chain[:-1]:
            h = _ext.pm_linear(h, W, b, _ext.PM_HIDDEN, n)      # relu(h @ W^T + b), fp16 pair out
        W, b = chain[-1]
        out, (hi, lo) = _ext.pm_linear(h, W, b, _ext.PM_OUT_CM, n)     # fp32 channel-major for the API + pm pair
        return attach_pm(out, hi.view(B, n, -1), lo.view(B, n, -1))


class PointnetLFPModuleMSG(nn.Module):
    """Learnable feature propagation (group features1 around xyz2, MLP, pool, post-MLP)."""

    def __init__(self, *, mlps: List[List[int]], radii: List[float], nsamples: List[int],
                 post_mlp: List[int], bn: bool = True, use_xyz: bool = True,
                 sample_uniformly: bool = False):
        super().__init__()
        assert len(mlps) == len(nsamples) == len(radii)
        self.post_mlp = pt_utils.SharedMLP(post_mlp, bn=bn)
        self.groupers, self.mlps = _build_groupers(0, radii, nsamples, mlps, bn, use_xyz,
                                                   sample_uniformly)

    def forward(self, xyz2: torch.Tensor, xyz1: torch.Tensor, features2: torch.Tensor,
                features1: torch.Tensor) -> torch.Tensor:
        outs = []
        for grouper, mlp in zip(self.groupers, self.mlps):
            new_features = _pool_max(mlp(grouper(xyz1, xyz2, features1)))
            if features2 is not None:
                new_features = torch.cat([new_features, features2], dim=1)
            outs.append(self.post_mlp(new_features.unsqueeze(-1)))
        return torch.cat(outs, dim=1).squeeze(-1)
