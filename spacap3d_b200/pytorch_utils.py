"""Same public API and parameter tree as the reference's lib/pointnet2/pytorch_utils.py
(SharedMLP :11-36, _BNBase :39-64, _ConvBase :67-120, Conv1d/2d/3d :123-233, FC :236-268,
set_bn_momentum_default / BNMomentumScheduler :270-296), written from scratch.

The state-dict contract (SURVEY F11) is what matters: a SharedMLP owns `layer{i}` children, each
a sequential block with `conv` (bias only when there is no BN), `bn` (itself a block with one
child `bn`) and `activation`, so keys read `...layer0.conv.weight`, `...layer0.bn.bn.running_mean`.
"""
import torch
import torch.distributed as dist
import torch.nn as nn
import torch.nn.functional as F

# Training mode: run BatchNorm2d + ReLU of a conv block through the fused sm_100a kernels (csrc/bn_relu.cu)
# instead of cuDNN batch-norm + a separate ReLU pass.  Same parameters, buffers and results (fp32, within
# summation-order rounding); set to False to get the plain module sequence.  A BatchNorm converted to
# nn.SyncBatchNorm runs the synced variants of the same kernels when torch's SyncBatchNorm would synchronise.
# Under torch.autocast(dtype=torch.bfloat16) the convolution returns bf16 and the kernels' bf16 twins run: bf16
# activations, fp32 arithmetic and fp32 BatchNorm parameters and statistics, as torch's own bf16 sequence.
FUSED_BN_RELU_TRAINING = True

# storage dtypes of a conv output the fused kernels take; anything else (fp16 autocast, fp64) runs torch's modules
_FUSED_DTYPES = (torch.float32, torch.bfloat16)


class _BnReluTrain(torch.autograd.Function):
    """z = relu(batch_norm(y, training=True)); saves y and the batch statistics, recomputes the ReLU mask.  With a
    process `group`, the statistics are those of every rank of it (torch.nn.SyncBatchNorm semantics): one exchange of
    (n, mean, M2) per channel in the forward and one of (n, sum dm, sum dm * xhat) in the backward."""

    @staticmethod
    def forward(ctx, y, gamma, beta, running_mean, running_var, momentum, eps, group):
        from . import _ext
        if group is None:
            z, mean, invstd = _ext.bn_relu_train_forward(y, gamma, beta, running_mean, running_var, momentum, eps)
        else:
            rows, mine = _exchange_rows(y.shape[1], group, y.device)
            _ext.bn_relu_sync_stats(y, mine)
            z, mean, invstd = _ext.bn_relu_sync_forward(y, gamma, beta, running_mean, running_var, momentum, eps,
                                                        _all_gather_rows(rows, group))
        ctx.save_for_backward(y, gamma, beta, mean, invstd)
        ctx.group = group
        return z

    @staticmethod
    def backward(ctx, dz):
        from . import _ext
        y, gamma, beta, mean, invstd = ctx.saved_tensors
        dz = dz.contiguous()
        if ctx.group is None:
            dy, dgamma, dbeta = _ext.bn_relu_train_backward(dz, y, gamma, beta, mean, invstd)
        else:
            rows, mine = _exchange_rows(y.shape[1], ctx.group, y.device)
            dgamma, dbeta = _ext.bn_relu_sync_backward_reduce(dz, y, gamma, beta, mean, invstd, mine)
            dy = _ext.bn_relu_sync_backward(dz, y, gamma, beta, mean, invstd, _all_gather_rows(rows, ctx.group))
        return dy, dgamma, dbeta, None, None, None, None, None


def _max_pool_last(x):
    """The SA module's pooling (pointnet2_modules.py:256-259) for the shapes the fused kernel does not take."""
    return torch.nn.functional.max_pool2d(x, kernel_size=[1, x.size(3)]).squeeze(-1)


class _BnReluMaxPoolTrain(torch.autograd.Function):
    """pooled = max_k relu(batch_norm(y, training=True))[..., k] for y (B,C,npoint,nsample); `group` as in
    _BnReluTrain."""

    @staticmethod
    def forward(ctx, y, gamma, beta, running_mean, running_var, momentum, eps, group):
        from . import _ext
        if group is None:
            pooled, argmax, ymax, mean, invstd = _ext.bn_relu_maxpool_train_forward(
                y, gamma, beta, running_mean, running_var, momentum, eps)
        else:
            rows, mine = _exchange_rows(y.shape[1], group, y.device)
            _ext.bn_relu_sync_stats(y, mine)
            pooled, argmax, ymax, mean, invstd = _ext.bn_relu_maxpool_sync_forward(
                y, gamma, beta, running_mean, running_var, momentum, eps, _all_gather_rows(rows, group))
        ctx.save_for_backward(y, gamma, beta, mean, invstd, argmax, ymax)
        ctx.group = group
        return pooled

    @staticmethod
    def backward(ctx, dpool):
        from . import _ext
        y, gamma, beta, mean, invstd, argmax, ymax = ctx.saved_tensors
        dpool = dpool.contiguous()
        if ctx.group is None:
            dy, dgamma, dbeta = _ext.bn_relu_maxpool_train_backward(dpool, argmax, ymax, y, gamma, beta, mean, invstd)
        else:
            rows, mine = _exchange_rows(y.shape[1], ctx.group, y.device)
            dgamma, dbeta = _ext.bn_relu_maxpool_sync_backward_reduce(dpool, ymax, y, gamma, beta, mean, invstd, mine)
            dy = _ext.bn_relu_maxpool_sync_backward(dpool, argmax, ymax, y, gamma, beta, mean, invstd,
                                                    _all_gather_rows(rows, ctx.group))
        return dy, dgamma, dbeta, None, None, None, None, None


def _exchange_rows(C, group, device):
    """Zeroed (world, C, BN_SYNC_K) f64 buffer and this rank's row of it."""
    from . import _ext
    rows = torch.zeros((dist.get_world_size(group), C, _ext.BN_SYNC_K), dtype=torch.float64, device=device)
    return rows, rows[dist.get_rank(group)]


def _all_gather_rows(rows, group):
    """Every rank filled only its own row of a zeroed buffer, so the SUM all-reduce is an exact all-gather (no
    floating-point addition ever meets two non-zero terms); the rows are then combined in rank order on the device."""
    dist.all_reduce(rows, op=dist.ReduceOp.SUM, group=group)
    return rows


def _sync_group(bn):
    """The process group a training-mode nn.SyncBatchNorm synchronises over, or None when it would not (not a
    SyncBatchNorm, torch.distributed not initialised, or a group of one rank): torch's own rule."""
    if not (isinstance(bn, nn.SyncBatchNorm) and dist.is_available() and dist.is_initialized()):
        return None
    group = bn.process_group if bn.process_group is not None else dist.group.WORLD
    return group if dist.get_world_size(group) > 1 else None


_CONV = {1: nn.Conv1d, 2: nn.Conv2d, 3: nn.Conv3d}
_NORM = {1: nn.BatchNorm1d, 2: nn.BatchNorm2d, 3: nn.BatchNorm3d}


class _BNBase(nn.Sequential):
    def __init__(self, in_size, batch_norm=None, name=""):
        super().__init__()
        norm = batch_norm(in_size)
        nn.init.constant_(norm.weight, 1.0)
        nn.init.constant_(norm.bias, 0)
        self.add_module(name + "bn", norm)


class BatchNorm1d(_BNBase):
    def __init__(self, in_size, *, name=""):
        super().__init__(in_size, batch_norm=_NORM[1], name=name)


class BatchNorm2d(_BNBase):
    def __init__(self, in_size, name=""):
        super().__init__(in_size, batch_norm=_NORM[2], name=name)


class BatchNorm3d(_BNBase):
    def __init__(self, in_size, name=""):
        super().__init__(in_size, batch_norm=_NORM[3], name=name)


class _ConvBase(nn.Sequential):
    """[bn, act,] conv [, bn, act] depending on `preact`; conv bias only without BN."""

    def __init__(self, in_size, out_size, kernel_size, stride, padding, activation, bn, init,
                 conv=None, batch_norm=None, bias=True, preact=False, name=""):
        super().__init__()
        use_bias = bias and not bn
        conv_unit = conv(in_size, out_size, kernel_size=kernel_size, stride=stride,
                         padding=padding, bias=use_bias)
        init(conv_unit.weight)
        if use_bias:
            nn.init.constant_(conv_unit.bias, 0)
        norm_unit = batch_norm(in_size if preact else out_size) if bn else None

        def _norm_act():
            if norm_unit is not None:
                self.add_module(name + "bn", norm_unit)
            if activation is not None:
                self.add_module(name + "activation", activation)

        if preact:
            _norm_act()
        self.add_module(name + "conv", conv_unit)
        if not preact:
            _norm_act()
        # conv -> BatchNorm2d -> ReLU is the only arrangement SpaCap3D instantiates; remember it for forward()
        self._fusable = (not preact and norm_unit is not None and isinstance(activation, nn.ReLU)
                         and isinstance(conv_unit, nn.Conv2d))
        self._conv_name, self._bn_name = name + "conv", name + "bn"   # names, not modules: no second registration

    def _fused_training_ok(self, x):
        """Everything but the conv output's dtype, which forward() checks once the conv has run (autocast decides
        it).  The BatchNorm's parameters must be fp32: a model cast wholesale with .bfloat16() keeps torch's."""
        if not (self._fusable and FUSED_BN_RELU_TRAINING and self.training and x.is_cuda and torch.is_grad_enabled()):
            return False
        bn = getattr(self, self._bn_name)[0]
        return (bn.training and bn.affine and bn.track_running_stats and bn.momentum is not None
                and bn.weight.dtype == torch.float32 and bn.running_mean.dtype == torch.float32)

    def forward(self, x, max_pool_last_dim=False):
        """max_pool_last_dim=True additionally takes the max over the last axis (the SA module's
        F.max_pool2d(kernel=[1, nsample]) + squeeze) and returns (B, C, npoint)."""
        conv = getattr(self, self._conv_name)
        if x.shape[1] > conv.in_channels:
            # the caller appended all-zero channels for 16-byte-aligned GEMM rows (QueryAndGroup pad_channels_to):
            # the same convolution with matching zero weight columns; autograd slices the weight gradient back
            extra = x.shape[1] - conv.in_channels
            w = F.pad(conv.weight, (0, 0) * (conv.weight.dim() - 2) + (0, extra))
            run_conv = lambda t: F.conv2d(t, w, conv.bias, conv.stride, conv.padding)   # noqa: E731
        else:
            run_conv = conv
        if self._fused_training_ok(x):
            bn = getattr(self, self._bn_name)[0]
            # the kernels take any batch, so whether they run depends only on the module, C and nsample, never on this
            # rank's share of the batch: with SyncBatchNorm all ranks issue the same collectives
            y = run_conv(x).contiguous()
            if y.dtype not in _FUSED_DTYPES:
                out = y
                for name, mod in self.named_children():      # conv -> bn -> activation; the conv has run
                    if name != self._conv_name:
                        out = mod(out)
                return _max_pool_last(out) if max_pool_last_dim else out
            args = (y, bn.weight, bn.bias, bn.running_mean, bn.running_var, float(bn.momentum), float(bn.eps),
                    _sync_group(bn))
            if max_pool_last_dim and y.dim() == 4 and y.shape[3] in (16, 32, 64):
                out = _BnReluMaxPoolTrain.apply(*args)
            else:
                out = _BnReluTrain.apply(*args)
                if max_pool_last_dim:
                    out = _max_pool_last(out)
            if bn.num_batches_tracked is not None:
                bn.num_batches_tracked.add_(1)
            return out
        if run_conv is not conv:
            out = x
            for name, mod in self.named_children():
                out = run_conv(out) if name == self._conv_name else mod(out)
        else:
            out = super().forward(x)
        return _max_pool_last(out) if max_pool_last_dim else out


def _make_conv(dim, wrapper):
    ones, zeros = (1,) * dim, (0,) * dim
    if dim == 1:
        ones, zeros = 1, 0

    class _Conv(_ConvBase):
        def __init__(self, in_size, out_size, *, kernel_size=ones, stride=ones, padding=zeros,
                     activation=nn.ReLU(inplace=True), bn=False, init=nn.init.kaiming_normal_,
                     bias=True, preact=False, name=""):
            super().__init__(in_size, out_size, kernel_size, stride, padding, activation, bn, init,
                             conv=_CONV[dim], batch_norm=wrapper, bias=bias, preact=preact,
                             name=name)

    _Conv.__name__ = _Conv.__qualname__ = "Conv%dd" % dim
    return _Conv


Conv1d = _make_conv(1, BatchNorm1d)
Conv2d = _make_conv(2, BatchNorm2d)
Conv3d = _make_conv(3, BatchNorm3d)


class SharedMLP(nn.Sequential):
    """Stack of 1x1 Conv2d (+BN +ReLU) blocks named layer0, layer1, ...  (reference :11-36)."""

    def __init__(self, args, *, bn=False, activation=nn.ReLU(inplace=True), preact=False,
                 first=False, name=""):
        super().__init__()
        for i, (cin, cout) in enumerate(zip(args[:-1], args[1:])):
            plain = first and preact and i == 0   # the very first pre-activation block is bare
            self.add_module(name + "layer{}".format(i),
                            Conv2d(cin, cout, bn=bn and not plain,
                                   activation=None if plain else activation, preact=preact))

    def forward_max_pooled(self, x):
        """self(x) followed by the max over the last axis, with the last block's BatchNorm + ReLU + max
        fused in training mode (csrc/bn_relu.cu); returns (B, C_out, npoint)."""
        blocks = list(self.children())
        for blk in blocks[:-1]:
            x = blk(x)
        return blocks[-1](x, max_pool_last_dim=True)


class FC(nn.Sequential):
    def __init__(self, in_size, out_size, *, activation=nn.ReLU(inplace=True), bn=False, init=None,
                 preact=False, name=""):
        super().__init__()
        fc = nn.Linear(in_size, out_size, bias=not bn)
        if init is not None:
            init(fc.weight)
        if not bn:
            nn.init.constant_(fc.bias, 0)

        def _norm_act(width):
            if bn:
                self.add_module(name + "bn", BatchNorm1d(width))
            if activation is not None:
                self.add_module(name + "activation", activation)

        if preact:
            _norm_act(in_size)
        self.add_module(name + "fc", fc)
        if not preact:
            _norm_act(out_size)


def set_bn_momentum_default(bn_momentum):
    def fn(m):
        if isinstance(m, (nn.BatchNorm1d, nn.BatchNorm2d, nn.BatchNorm3d)):
            m.momentum = bn_momentum
    return fn


class BNMomentumScheduler(object):
    """Sets every BN layer's momentum to bn_lambda(epoch) (used by lib/solver.py:19)."""

    def __init__(self, model, bn_lambda, last_epoch=-1, setter=set_bn_momentum_default):
        if not isinstance(model, nn.Module):
            raise RuntimeError("Class '{}' is not a PyTorch nn Module".format(type(model).__name__))
        self.model = model
        self.setter = setter
        self.lmbd = bn_lambda
        self.step(last_epoch + 1)
        self.last_epoch = last_epoch

    def step(self, epoch=None):
        if epoch is None:
            epoch = self.last_epoch + 1
        self.last_epoch = epoch
        self.model.apply(self.setter(self.lmbd(epoch)))
