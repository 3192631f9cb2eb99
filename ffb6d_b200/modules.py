"""``nn.Module`` twins of the reference's 1x1 layers and RandLA blocks, on this package's kernels, with
the reference's parameter names -- a maintainer can import-swap them and load published checkpoints.

* :class:`Conv2d` -- ``pt_utils.Conv2d`` of the fusion layers (models/pytorch_utils.py:168-201:
  ``conv`` -> ``normlayer.bn`` -> ``activation``; BatchNorm2d defaults eps 1e-5, momentum 0.1, ReLU).
* :class:`RandLAConv2d` -- RandLA's flavour (models/RandLA/pytorch_utils.py:163-197: ``conv`` -> ``bn.bn``
  -> ``activation``; eps 1e-6, momentum 0.99, LeakyReLU(0.2)).
* :class:`Att_pooling`, :class:`Building_block`, :class:`Dilated_res_block` -- models/RandLA/RandLANet.py:170-250.

Both modes run on the CUDA library:

* ``eval()``: one fused tensor-core kernel per layer (``ffb6d_fusion_mlp_fwd_ex``: concat + conv + folded
  BatchNorm + activation).
* ``train()``: batch-statistics BatchNorm and autograd -- forward = GEMM (tcgen05) + ``ffb6d_bn_train_fwd``
  (running statistics updated like ``nn.BatchNorm2d``); backward = ``ffb6d_bn_train_bwd``, weight gradient
  ``ffb6d_fusion_mlp_wgrad`` (tcgen05, split-K), input gradient = the forward GEMM with the transposed
  weight; neighbour gathers and attentive pooling have their own backward kernels.

A layer accepts its input as one tensor or as the two halves of a concat (``layer(x1, x2)`` ==
``layer(torch.cat((x1, x2), 1))`` without materialising the concat, models/ffb6d.py:251-262).

Synchronised BatchNorm: the reference trains with every BatchNorm converted to SyncBN (train_ycb.py:568).
``torch.nn.SyncBatchNorm.convert_sync_batchnorm(model)`` works on these modules and keeps the state-dict keys.
A layer whose ``bn`` child is an ``nn.SyncBatchNorm`` then decides like torch does: in training mode, with
``torch.distributed`` initialised and more than one rank in ``bn.process_group`` (default WORLD), it normalises
with the statistics of the global batch -- one all-reduce of the fp64 per-channel sums and the local element
count in the forward (``ffb6d_bn_train_stats`` / ``_apply``), one in the backward (``ffb6d_bn_train_bwd_stats`` /
``_bwd_apply``); the global count is read back to the host, one synchronisation per layer.  Running statistics
come out identical on every rank; gamma / beta gradients are the local sums, which DDP averages.  Every rank
needs at least one frame.  Otherwise (eval mode, one rank, no process group) the layer runs exactly as unconverted.
"""
import torch
import torch.distributed as dist
import torch.nn as nn
import torch.nn.functional as F_

from . import ops
from ._lib import lib, check

_ACT_NONE, _ACT_RELU, _ACT_LEAKY = 0, 1, 2


def _act_code(activation):
    if activation is None:
        return _ACT_NONE, 0.0
    if isinstance(activation, nn.ReLU):
        return _ACT_RELU, 0.0
    if isinstance(activation, nn.LeakyReLU):
        return _ACT_LEAKY, float(activation.negative_slope)
    raise ValueError("activation must be None, nn.ReLU or nn.LeakyReLU, got %r" % (activation,))


_const_cache = {}


def _ones_zeros(n, device):
    key = (n, device)
    if key not in _const_cache:
        _const_cache[key] = (torch.ones(n, device=device), torch.zeros(n, device=device))
    return _const_cache[key]


def _gemm(x1, x2, w2d):
    """z = W . cat(x1, x2), no affine, no activation (tcgen05 kernel)."""
    one, zero = _ones_zeros(w2d.shape[0], x1.device)
    return ops.fusion_mlp(x1, x2, w2d, one, zero, relu=False)


class _ConvBnActTrain(torch.autograd.Function):
    """conv1x1(cat(x1, x2)) -> [BatchNorm with batch statistics] -> activation, with its backward.
    ``group``: a process group to take the BatchNorm statistics over (SyncBatchNorm), or None for this rank's."""

    @staticmethod
    def forward(ctx, x1, x2, weight, bias, gamma, beta, running_mean, running_var, eps, momentum, act, slope, has_bn,
                group=None):
        x1 = x1.contiguous()
        x2 = x2.contiguous() if x2 is not None else None
        B, C1 = x1.shape[0], x1.shape[1]
        C2 = x2.shape[1] if x2 is not None else 0
        w2d = weight.reshape(weight.shape[0], -1).contiguous()
        Co = w2d.shape[0]
        if bias is not None:     # conv bias (only without BatchNorm): the GEMM epilogue's shift
            one, _ = _ones_zeros(Co, x1.device)
            z = ops.fusion_mlp(x1, x2, w2d, one, bias, relu=False)
        else:
            z = _gemm(x1, x2, w2d)
        P = z.numel() // (B * Co)
        stats = count = None
        if has_bn:
            stats = torch.empty((Co, 4), dtype=torch.float32, device=z.device)
            y = torch.empty_like(z)
            nbytes = int(lib.ffb6d_bn_workspace_bytes(Co, P))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=z.device)
            affine = (gamma.data_ptr() if gamma is not None else None, beta.data_ptr() if beta is not None else None,
                      float(eps), float(momentum), running_mean.data_ptr() if running_mean is not None else None,
                      running_var.data_ptr() if running_var is not None else None, int(act), float(slope),
                      stats.data_ptr(), y.data_ptr())
            with torch.cuda.device(z.device):
                if group is None:
                    check(lib.ffb6d_bn_train_fwd(z.data_ptr(), B, Co, P, *affine, ws.data_ptr(), nbytes,
                                                 ops._stream(z.device)))
                else:
                    # [(sum z, sum z^2) per channel, local element count], summed over the group; the counts
                    # may differ between ranks
                    sums = torch.empty(2 * Co + 1, dtype=torch.float64, device=z.device)
                    check(lib.ffb6d_bn_train_stats(z.data_ptr(), B, Co, P, sums.data_ptr(), ws.data_ptr(), nbytes,
                                                   ops._stream(z.device)))
                    sums[2 * Co] = float(B * P)
                    dist.all_reduce(sums, group=group)
                    count = float(sums[2 * Co])
                    check(lib.ffb6d_bn_train_apply(z.data_ptr(), B, Co, P, sums.data_ptr(), count, *affine,
                                                   ops._stream(z.device)))
        elif act == _ACT_RELU:
            y = torch.relu(z)
        elif act == _ACT_LEAKY:
            y = F_.leaky_relu(z, slope)
        else:
            y = z
        ctx.save_for_backward(x1, x2, w2d, z, stats, gamma)
        ctx.meta = (B, C1, C2, Co, P, int(act), float(slope), bool(has_bn), bias is not None, tuple(weight.shape))
        ctx.sync = (group, count)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        x1, x2, w2d, z, stats, gamma = ctx.saved_tensors
        B, C1, C2, Co, P, act, slope, has_bn, has_bias, wshape = ctx.meta
        group, count = ctx.sync
        gy = gy.contiguous()
        dev = z.device
        ggamma = gbeta = gbias = None
        with torch.cuda.device(dev):
            if has_bn:
                dz = torch.empty_like(z)
                ggamma = torch.empty(Co, dtype=torch.float32, device=dev)
                gbeta = torch.empty(Co, dtype=torch.float32, device=dev)
                nbytes = int(lib.ffb6d_bn_workspace_bytes(Co, P))
                ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                if group is None:
                    check(lib.ffb6d_bn_train_bwd(z.data_ptr(), gy.data_ptr(), stats.data_ptr(), B, Co, P, act, slope,
                                                 ggamma.data_ptr(), gbeta.data_ptr(), dz.data_ptr(), ws.data_ptr(),
                                                 nbytes, ops._stream(dev)))
                else:
                    sums = torch.empty(2 * Co, dtype=torch.float64, device=dev)
                    check(lib.ffb6d_bn_train_bwd_stats(z.data_ptr(), gy.data_ptr(), stats.data_ptr(), B, Co, P, act,
                                                       slope, sums.data_ptr(), ggamma.data_ptr(), gbeta.data_ptr(),
                                                       ws.data_ptr(), nbytes, ops._stream(dev)))
                    dist.all_reduce(sums, group=group)
                    check(lib.ffb6d_bn_train_bwd_apply(z.data_ptr(), gy.data_ptr(), stats.data_ptr(), sums.data_ptr(),
                                                       count, B, Co, P, act, slope, dz.data_ptr(), ops._stream(dev)))
            elif act != _ACT_NONE:
                dz = torch.empty_like(z)
                check(lib.ffb6d_act_bwd(z.data_ptr(), gy.data_ptr(), z.numel(), act, slope, dz.data_ptr(), ops._stream(dev)))
            else:
                dz = gy
            gw = None
            if ctx.needs_input_grad[2]:
                gw = torch.empty((Co, C1 + C2), dtype=torch.float32, device=dev)
                check(lib.ffb6d_fusion_mlp_wgrad(dz.data_ptr(), x1.data_ptr(), C1, x2.data_ptr() if x2 is not None else None,
                                                 C2, B, Co, P, gw.data_ptr(), ops._stream(dev)))
                gw = gw.reshape(wshape)
        if has_bias:
            gbias = dz.reshape(B, Co, -1).sum(dim=(0, 2))
        # input gradients: dX = W^T . dz, one GEMM per half of the concat
        gx1 = gx2 = None
        if ctx.needs_input_grad[0]:
            gx1 = _gemm(dz, None, w2d[:, :C1].t().contiguous()).reshape(x1.shape)
        if x2 is not None and ctx.needs_input_grad[1]:
            gx2 = _gemm(dz, None, w2d[:, C1:].t().contiguous()).reshape(x2.shape)
        if gamma is None:
            ggamma = None
        return gx1, gx2, gw, gbias, ggamma, gbeta, None, None, None, None, None, None, None, None


def _sync_group(bn):
    """The process group a training-mode ``nn.SyncBatchNorm`` takes its statistics over, decided as
    ``nn.SyncBatchNorm.forward`` decides; None for any other BatchNorm or when there is nothing to sync with."""
    if not isinstance(bn, nn.SyncBatchNorm) or not (dist.is_available() and dist.is_initialized()):
        return None
    group = bn.process_group if bn.process_group is not None else dist.group.WORLD
    return group if dist.get_world_size(group) > 1 else None


class _BNWrap(nn.Sequential):
    """The reference's ``_BNBase``: a Sequential holding one BatchNorm2d named ``bn``."""

    def __init__(self, channels, eps, momentum, dims=2):
        super().__init__()
        self.add_module("bn", (nn.BatchNorm2d if dims == 2 else nn.BatchNorm1d)(channels, eps=eps, momentum=momentum))
        nn.init.constant_(self[0].weight, 1.0)
        nn.init.constant_(self[0].bias, 0)


class _ConvBase(nn.Module):
    _bn_name = "normlayer"
    _bn_eps, _bn_momentum = 1e-5, 0.1

    _dims = 2

    def __init__(self, in_size, out_size, kernel_size=(1, 1), activation=None, bn=False, init=nn.init.kaiming_normal_,
                 bias=True, name=""):
        super().__init__()
        ks = (kernel_size,) if isinstance(kernel_size, int) else tuple(kernel_size)
        if any(k != 1 for k in ks):
            raise ValueError("only the 1x1 layers of the fusion / RandLA path are implemented here")
        bias = bias and (not bn)
        # holds the parameters under the reference's names; the arithmetic runs in the CUDA library
        conv_unit = (nn.Conv2d(in_size, out_size, kernel_size=(1, 1), bias=bias) if self._dims == 2
                     else nn.Conv1d(in_size, out_size, kernel_size=1, bias=bias))
        init(conv_unit.weight)
        if bias:
            nn.init.constant_(conv_unit.bias, 0)
        self._names = (name + "conv", name + self._bn_name)
        self.add_module(name + "conv", conv_unit)
        self.has_bn = bool(bn)
        if bn:
            self.add_module(name + self._bn_name, _BNWrap(out_size, self._bn_eps, self._bn_momentum, self._dims))
        if activation is not None:
            self.add_module(name + "activation", activation)
        self.act, self.slope = _act_code(activation)
        self._packed = None      # (weight version, PackedWeight, scale, shift) of the eval path

    @property
    def _conv(self):
        return getattr(self, self._names[0])

    @property
    def _bn(self):
        return getattr(self, self._names[1]).bn if self.has_bn else None

    def _eval_pack(self):
        conv, bn = self._conv, self._bn
        ver = (conv.weight._version, conv.weight.data_ptr(), bn.weight._version if bn is not None else 0,
               bn.running_mean._version if bn is not None else 0)
        if self._packed is None or self._packed[0] != ver:
            w = conv.weight.detach()
            if bn is not None:
                scale, shift = ops.fold_batchnorm(bn)
            else:
                scale = torch.ones(w.shape[0], device=w.device)
                shift = conv.bias.detach().float() if conv.bias is not None else torch.zeros_like(scale)
            self._packed = (ver, ops.fusion_mlp_pack(w), scale, shift)
        return self._packed[1:]

    def forward(self, x, x2=None):
        if self._dims == 1:     # [B, C, N] layers run as [B, C, N, 1]
            return self._forward(x.unsqueeze(3), x2.unsqueeze(3) if x2 is not None else None).squeeze(3)
        return self._forward(x, x2)

    def _forward(self, x, x2=None):
        conv, bn = self._conv, self._bn
        need_grad = torch.is_grad_enabled() and (x.requires_grad or conv.weight.requires_grad or
                                                 (x2 is not None and x2.requires_grad))
        if self.training and bn is not None:
            if bn.track_running_stats and bn.num_batches_tracked is not None:
                bn.num_batches_tracked += 1
            return _ConvBnActTrain.apply(x, x2, conv.weight, None, bn.weight, bn.bias, bn.running_mean, bn.running_var,
                                         bn.eps, bn.momentum if bn.momentum is not None else 0.1, self.act, self.slope, True,
                                         _sync_group(bn))
        if need_grad and bn is None:
            return _ConvBnActTrain.apply(x, x2, conv.weight, conv.bias, None, None, None, None, 0.0, 0.0, self.act,
                                         self.slope, False)
        if need_grad:
            # eval-mode BatchNorm under autograd (fine-tuning with frozen statistics): GEMM with its backward,
            # then the per-channel affine and the activation as differentiable elementwise torch ops
            z = _ConvBnActTrain.apply(x, x2, conv.weight, None, None, None, None, None, 0.0, 0.0, _ACT_NONE, 0.0, False)
            y = F_.batch_norm(z, bn.running_mean, bn.running_var, bn.weight, bn.bias, False, 0.0, bn.eps)
            if self.act == _ACT_RELU:
                return torch.relu(y)
            return F_.leaky_relu(y, self.slope) if self.act == _ACT_LEAKY else y
        packed, scale, shift = self._eval_pack()
        return ops.fusion_mlp(x, x2, packed, scale, shift, relu=(self.act == _ACT_RELU),
                              negative_slope=self.slope if self.act == _ACT_LEAKY else None)


class Conv2d(_ConvBase):
    """``pt_utils.Conv2d`` of FFB6D's fusion layers (models/pytorch_utils.py:168-201), 1x1 only.
    State-dict keys: ``conv.weight``, ``normlayer.bn.{weight,bias,running_mean,running_var,num_batches_tracked}``."""

    def __init__(self, in_size, out_size, kernel_size=(1, 1), stride=(1, 1), padding=(0, 0), dilation=(1, 1),
                 activation=nn.ReLU(inplace=True), bn=False, init=nn.init.kaiming_normal_, bias=True, preact=False, name=""):
        if preact or tuple(stride) != (1, 1) or tuple(padding) != (0, 0) or tuple(dilation) != (1, 1):
            raise ValueError("only plain 1x1 layers (no preact / stride / padding / dilation) are implemented here")
        super().__init__(in_size, out_size, kernel_size, activation, bn, init, bias, name)


class RandLAConv2d(_ConvBase):
    """RandLA's ``pt_utils.Conv2d`` (models/RandLA/pytorch_utils.py:163-197), 1x1 only.
    State-dict keys: ``conv.weight``, ``bn.bn.{weight,bias,running_mean,running_var,num_batches_tracked}``."""
    _bn_name = "bn"
    _bn_eps, _bn_momentum = 1e-6, 0.99

    def __init__(self, in_size, out_size, *, kernel_size=(1, 1), stride=(1, 1), padding=(0, 0),
                 activation=nn.LeakyReLU(negative_slope=0.2, inplace=True), bn=False, init=nn.init.kaiming_normal_,
                 bias=True, preact=False, name="", instance_norm=False):
        if preact or instance_norm or tuple(stride) != (1, 1) or tuple(padding) != (0, 0):
            raise ValueError("only plain 1x1 layers are implemented here")
        super().__init__(in_size, out_size, kernel_size, activation, bn, init, bias, name)


class Conv1d(_ConvBase):
    """``pt_utils.Conv1d`` of FFB6D's prediction heads (models/pytorch_utils.py:132-165), kernel size 1: input
    ``[B, C, N]``.  State-dict keys as :class:`Conv2d` (``conv.weight`` is ``[Co, Ci, 1]``)."""
    _dims = 1

    def __init__(self, in_size, out_size, kernel_size=1, stride=1, padding=0, dilation=1,
                 activation=nn.ReLU(inplace=True), bn=False, init=nn.init.kaiming_normal_, bias=True, preact=False, name=""):
        if preact or stride != 1 or padding != 0 or dilation != 1:
            raise ValueError("only plain kernel-size-1 layers are implemented here")
        super().__init__(in_size, out_size, kernel_size, activation, bn, init, bias, name)


class RandLAConv1d(_ConvBase):
    """RandLA's ``pt_utils.Conv1d`` (``fc0`` of the network, models/RandLA/RandLANet.py:16), kernel size 1."""
    _dims = 1
    _bn_name = "bn"
    _bn_eps, _bn_momentum = 1e-6, 0.99

    def __init__(self, in_size, out_size, *, kernel_size=1, stride=1, padding=0,
                 activation=nn.LeakyReLU(negative_slope=0.2, inplace=True), bn=False, init=nn.init.kaiming_normal_,
                 bias=True, preact=False, name="", instance_norm=False):
        if preact or instance_norm or stride != 1 or padding != 0:
            raise ValueError("only plain kernel-size-1 layers are implemented here")
        super().__init__(in_size, out_size, kernel_size, activation, bn, init, bias, name)


# ----------------------------------------------------------------------------------------- RandLA blocks
class _AttPool(torch.autograd.Function):
    @staticmethod
    def forward(ctx, f1, f2, att):
        out = ops.att_pool(f1, f2, att)
        ctx.save_for_backward(f1.contiguous(), f2.contiguous() if f2 is not None else None, att.contiguous())
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        f1, f2, att = ctx.saved_tensors
        B, C1, N, K = f1.shape
        C2 = f2.shape[1] if f2 is not None else 0
        g = gout.contiguous()
        gf1, gatt = torch.empty_like(f1), torch.empty_like(att)
        gf2 = torch.empty_like(f2) if f2 is not None else None
        with torch.cuda.device(f1.device):
            check(lib.ffb6d_att_pool_bwd(f1.data_ptr(), C1, f2.data_ptr() if f2 is not None else None, C2, att.data_ptr(),
                                         g.data_ptr(), B, N, K, gf1.data_ptr(), gf2.data_ptr() if gf2 is not None else None,
                                         gatt.data_ptr(), ops._stream(f1.device)))
        return gf1, gf2, gatt


def _gather_cm(feature, neigh_idx):
    """feature [B,C,N,1] -> neighbours channel-major [B,C,N,K]: ``gather_neighbour`` + ``permute(0,3,1,2)``
    (RandLANet.py:200-203) as one K = 1 gather (differentiable)."""
    B, N, K = neigh_idx.shape
    g = ops.nearest_interpolation(feature, neigh_idx.reshape(B, N * K, 1))
    return g.reshape(B, feature.shape[1], N, K)


class Att_pooling(nn.Module):
    """models/RandLA/RandLANet.py:237-250.  ``forward(feature_set)`` as the reference, or
    ``forward(f_neighbours, f_xyz)`` = the same on their concat without materialising it."""

    def __init__(self, d_in, d_out):
        super().__init__()
        self.fc = nn.Conv2d(d_in, d_in, (1, 1), bias=False)
        self.mlp = RandLAConv2d(d_in, d_out, kernel_size=(1, 1), bn=True)
        self._fc_pack = None

    def _att(self, f1, f2):
        w = self.fc.weight
        if torch.is_grad_enabled() and (w.requires_grad or f1.requires_grad or (f2 is not None and f2.requires_grad)):
            return _ConvBnActTrain.apply(f1, f2, w, None, None, None, None, None, 0.0, 0.0, _ACT_NONE, 0.0, False)
        ver = (w._version, w.data_ptr())
        if self._fc_pack is None or self._fc_pack[0] != ver:
            self._fc_pack = (ver, ops.fusion_mlp_pack(w.detach()))
        one, zero = _ones_zeros(w.shape[0], f1.device)
        return ops.fusion_mlp(f1, f2, self._fc_pack[1], one, zero, relu=False)

    def forward(self, feature_set, f2=None):
        att = self._att(feature_set, f2)
        if torch.is_grad_enabled() and att.requires_grad:
            f_agg = _AttPool.apply(feature_set, f2, att)
        else:
            f_agg = ops.att_pool(feature_set, f2, att)
        return self.mlp(f_agg)


class Building_block(nn.Module):
    """models/RandLA/RandLANet.py:187-214 (local spatial encoding + two attentive poolings)."""

    def __init__(self, d_out):
        super().__init__()
        self.mlp1 = RandLAConv2d(10, d_out // 2, kernel_size=(1, 1), bn=True)
        self.att_pooling_1 = Att_pooling(d_out, d_out // 2)
        self.mlp2 = RandLAConv2d(d_out // 2, d_out // 2, kernel_size=(1, 1), bn=True)
        self.att_pooling_2 = Att_pooling(d_out, d_out)

    def forward(self, xyz, feature, neigh_idx):
        f_xyz = ops.relative_pos_encoding(xyz, neigh_idx, channel_major=True)     # [B,10,N,K]
        f_xyz = self.mlp1(f_xyz)
        f_pc_agg = self.att_pooling_1(_gather_cm(feature, neigh_idx), f_xyz)
        f_xyz = self.mlp2(f_xyz)
        return self.att_pooling_2(_gather_cm(f_pc_agg, neigh_idx), f_xyz)

    relative_pos_encoding = staticmethod(ops.relative_pos_encoding)
    gather_neighbour = staticmethod(ops.gather_neighbour)


class Dilated_res_block(nn.Module):
    """models/RandLA/RandLANet.py:170-184."""

    def __init__(self, d_in, d_out):
        super().__init__()
        self.mlp1 = RandLAConv2d(d_in, d_out // 2, kernel_size=(1, 1), bn=True)
        self.lfa = Building_block(d_out)
        self.mlp2 = RandLAConv2d(d_out, d_out * 2, kernel_size=(1, 1), bn=True, activation=None)
        self.shortcut = RandLAConv2d(d_in, d_out * 2, kernel_size=(1, 1), bn=True, activation=None)

    def forward(self, feature, xyz, neigh_idx):
        if not self.training and not torch.is_grad_enabled():
            from . import randla
            return randla.dilated_res_block(self.state_dict(), "", feature, xyz, neigh_idx)   # fused residual GEMM
        f_pc = self.mlp1(feature)
        f_pc = self.lfa(xyz, f_pc, neigh_idx)
        f_pc = self.mlp2(f_pc)
        shortcut = self.shortcut(feature)
        return F_.leaky_relu(f_pc + shortcut, negative_slope=0.2)
