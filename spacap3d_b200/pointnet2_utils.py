"""Same public API as the reference's lib/pointnet2/pointnet2_utils.py -- six autograd
Functions (furthest_point_sample :51-80, gather_operation :83-117, three_nn :120-149,
three_interpolate :152-206, grouping_operation :209-257, ball_query :260-291) plus
QueryAndGroup (:294-380), GroupAll (:383-429) and RandomDropout (:40-48) -- on top of this
package's sm_100a kernels (`_ext`, the stand-in for `pointnet2._ext`).

Autograd behaviour is kept: FPS / ball_query outputs are non-differentiable, three_nn returns no
gradients, gather / grouping / interpolate keep (idx, sizes) on ctx and scatter-add backwards.
"""
import torch
import torch.nn as nn
from torch.autograd import Function

from . import _ext
from . import pytorch_utils as pt_utils  # noqa: F401  (re-exported like the reference)


class RandomDropout(nn.Module):
    """Feature dropout with a random rate theta ~ U(0, p) and no rescaling.  (The reference's
    version calls a helper that does not exist, pointnet2_utils.py:48; this one works.)"""

    def __init__(self, p=0.5, inplace=False):
        super().__init__()
        self.p = p
        self.inplace = inplace

    def forward(self, X):
        if not self.training:
            return X
        theta = float(torch.empty(1).uniform_(0, self.p))
        keep = (torch.rand(X.shape[:2] + (1,) * (X.dim() - 2), device=X.device) >= theta).to(X.dtype)
        return X.mul_(keep) if self.inplace else X * keep


class FurthestPointSampling(Function):
    @staticmethod
    def forward(ctx, xyz, npoint):
        """xyz (B,N,3) -> (B,npoint) int32 indices of the greedy farthest-point subset."""
        fps_inds = _ext.furthest_point_sampling(xyz, npoint)
        ctx.mark_non_differentiable(fps_inds)
        return fps_inds

    @staticmethod
    def backward(ctx, a=None):
        return None, None


furthest_point_sample = FurthestPointSampling.apply


class GatherOperation(Function):
    @staticmethod
    def forward(ctx, features, idx):
        """features (B,C,N), idx (B,npoint) -> (B,C,npoint)"""
        _, C, N = features.size()
        ctx.for_backwards = (idx, C, N)
        return _ext.gather_points(features, idx)

    @staticmethod
    def backward(ctx, grad_out):
        idx, C, N = ctx.for_backwards
        return _ext.gather_points_grad(grad_out.contiguous(), idx, N), None


gather_operation = GatherOperation.apply


class ThreeNN(Function):
    @staticmethod
    def forward(ctx, unknown, known):
        """unknown (B,n,3), known (B,m,3) -> (dist (B,n,3) L2 distances, idx (B,n,3))"""
        dist2, idx = _ext.three_nn(unknown, known)
        return torch.sqrt(dist2), idx

    @staticmethod
    def backward(ctx, a=None, b=None):
        return None, None


three_nn = ThreeNN.apply


class ThreeInterpolate(Function):
    @staticmethod
    def forward(ctx, features, idx, weight):
        """features (B,c,m), idx (B,n,3), weight (B,n,3) -> (B,c,n)"""
        m = features.size(2)
        ctx.three_interpolate_for_backward = (idx, weight, m)
        return _ext.three_interpolate(features, idx, weight)

    @staticmethod
    def backward(ctx, grad_out):
        idx, weight, m = ctx.three_interpolate_for_backward
        return _ext.three_interpolate_grad(grad_out.contiguous(), idx, weight, m), None, None


three_interpolate = ThreeInterpolate.apply


class GroupingOperation(Function):
    @staticmethod
    def forward(ctx, features, idx):
        """features (B,C,N), idx (B,npoint,nsample) -> (B,C,npoint,nsample)"""
        N = features.size(2)
        ctx.for_backwards = (idx, N)
        return _ext.group_points(features, idx)

    @staticmethod
    def backward(ctx, grad_out):
        idx, N = ctx.for_backwards
        return _ext.group_points_grad(grad_out.contiguous(), idx, N), None


grouping_operation = GroupingOperation.apply


class BallQuery(Function):
    @staticmethod
    def forward(ctx, radius, nsample, xyz, new_xyz):
        """xyz (B,N,3), new_xyz (B,npoint,3) -> (B,npoint,nsample) int32.
        NB the argument swap: the extension takes (new_xyz, xyz) (reference :282)."""
        inds = _ext.ball_query(new_xyz, xyz, radius, nsample)
        ctx.mark_non_differentiable(inds)
        return inds

    @staticmethod
    def backward(ctx, a=None):
        return None, None, None, None


ball_query = BallQuery.apply


class QueryAndGroup(nn.Module):
    """ball query -> group xyz (relative to the centre, optionally / radius) -> group features
    -> concatenate xyz channels first (reference :294-380)."""

    def __init__(self, radius, nsample, use_xyz=True, ret_grouped_xyz=False, normalize_xyz=False,
                 sample_uniformly=False, ret_unique_cnt=False):
        super().__init__()
        self.radius, self.nsample, self.use_xyz = radius, nsample, use_xyz
        self.ret_grouped_xyz = ret_grouped_xyz
        self.normalize_xyz = normalize_xyz
        self.sample_uniformly = sample_uniformly
        self.ret_unique_cnt = ret_unique_cnt
        if self.ret_unique_cnt:
            assert self.sample_uniformly

    def forward(self, xyz, new_xyz, features=None, pad_channels_to=1, dtype=None):
        """xyz (B,N,3), new_xyz (B,npoint,3), features (B,C,N) -> (B,3+C,npoint,nsample).
        pad_channels_to = 4 (an extension the SA module uses in training) appends all-zero channels so that the
        channel count is a multiple of 4: 3 + 128 or 3 + 256 input channels make every row of the 1x1-conv GEMMs
        that follow 4 bytes short of 16-byte alignment, which sends cuDNN / cuBLAS to their slow `align1` kernels
        (14 % of a training step); the consumer pads its weight with matching zero columns.
        dtype = torch.bfloat16 (the SA module under bf16 autocast) groups the features cast to bf16 and casts the
        relative xyz before the concatenation: bit for bit the conv input autocast would produce, without an fp32
        copy of the grouped tensor (torch.cat promotes mixed inputs to fp32).  The returned grouped_xyz stays fp32."""
        if self.sample_uniformly:
            # the reference prints and exit(1)s here (:337-339); raise instead of killing the process
            raise NotImplementedError("sample_uniformly is a dead path in the reference")
        idx = ball_query(self.radius, self.nsample, xyz, new_xyz)
        grouped_xyz = grouping_operation(xyz.transpose(1, 2).contiguous(), idx)
        grouped_xyz -= new_xyz.transpose(1, 2).unsqueeze(-1)
        if self.normalize_xyz:
            grouped_xyz /= self.radius
        if features is not None:
            grouped_features = grouping_operation(features if dtype is None else features.to(dtype), idx)
            if self.use_xyz:
                xyz_part = grouped_xyz if dtype is None else grouped_xyz.to(dtype)
                parts = [xyz_part, grouped_features]
                extra = -(3 + grouped_features.shape[1]) % max(int(pad_channels_to), 1)
                if extra:
                    parts.append(xyz_part.new_zeros((xyz_part.shape[0], extra) + tuple(xyz_part.shape[2:])))
                new_features = torch.cat(parts, dim=1)
            else:
                new_features = grouped_features
        else:
            assert self.use_xyz, "Cannot have not features and not use xyz as a feature!"
            new_features = grouped_xyz
        ret = [new_features]
        if self.ret_grouped_xyz:
            ret.append(grouped_xyz)
        return ret[0] if len(ret) == 1 else tuple(ret)


class GroupAll(nn.Module):
    """npoint=None path: the whole cloud is one group (reference :383-429).  The reference never
    stores ret_grouped_xyz (AttributeError when reached, SURVEY a16); it is stored here."""

    def __init__(self, use_xyz=True, ret_grouped_xyz=False):
        super().__init__()
        self.use_xyz = use_xyz
        self.ret_grouped_xyz = ret_grouped_xyz

    def forward(self, xyz, new_xyz, features=None):
        """xyz (B,N,3), features (B,C,N) -> (B,3+C,1,N)"""
        grouped_xyz = xyz.transpose(1, 2).unsqueeze(2)
        if features is not None:
            grouped_features = features.unsqueeze(2)
            new_features = torch.cat([grouped_xyz, grouped_features], dim=1) if self.use_xyz \
                else grouped_features
        else:
            new_features = grouped_xyz
        return (new_features, grouped_xyz) if self.ret_grouped_xyz else new_features
