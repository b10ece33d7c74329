"""Drop-in for ``basicsr.models.ops.dcn`` (B2/B3 boundary of SURVEY §8b) on the B200 kernels.

Same public names, argument meaning, parameter names/shapes/initialisation and error behaviour as
/root/reference/basicsr/models/ops/dcn/deform_conv.py:
  ModulatedDeformConvFunction / modulated_deform_conv ... :111-185
  ModulatedDeformConv ................................. :295-342
  ModulatedDeformConvPack ............................. :345-390
and DCNv2Pack of /root/reference/basicsr/models/archs/arch_util.py:232-257.
  DeformConvFunction / deform_conv (DCNv1) ............. :12-108
  DeformConv / DeformConvPack ......................... :186-292

There is no CPU path and no fallback: CPU tensors raise NotImplementedError exactly like the
reference (deform_conv.py:133-134), and a missing libedvr_b200.so raises RuntimeError.
"""
import logging
import math

import torch
from torch import nn
from torch.autograd import Function
from torch.autograd.function import once_differentiable
from torch.nn.modules.utils import _pair, _single

from . import _lib as L
from . import ops

_MONITOR = ops.OffsetMonitor()       # deferred `offset_absmean > 50` warnings of the fused DCNv2Pack path


def _out_hw(H, W, kh, kw, stride, padding, dilation):
    return ((H + 2 * padding - (dilation * (kh - 1) + 1)) // stride + 1,
            (W + 2 * padding - (dilation * (kw - 1) + 1)) // stride + 1)


def _f32c(t):
    return t.detach().to(torch.float32).contiguous()


def _all_f64(*ts):
    """True when every given tensor (None = absent) is float64: such calls run the double-precision kernels."""
    return all(t is None or t.dtype == torch.float64 for t in ts)


def _f64c(t):
    return t.detach().contiguous()


class ModulatedDeformConvFunction(Function):

    @staticmethod
    def forward(ctx, input, offset, mask, weight, bias=None, stride=1, padding=0, dilation=1, groups=1,
                deformable_groups=1):
        ctx.stride, ctx.padding, ctx.dilation = stride, padding, dilation
        ctx.groups, ctx.deformable_groups = groups, deformable_groups
        ctx.with_bias = bias is not None
        if not input.is_cuda:
            raise NotImplementedError
        if weight.requires_grad or mask.requires_grad or offset.requires_grad or input.requires_grad:
            ctx.save_for_backward(input, offset, mask, weight, bias if ctx.with_bias else input.new_empty(1))
        ctx.f64 = _all_f64(input, offset, mask, weight, bias)
        if ctx.f64:
            return ops.mdcn_forward(_f64c(input), _f64c(offset), _f64c(mask), _f64c(weight),
                                    _f64c(bias) if ctx.with_bias else None, stride, padding, dilation, groups,
                                    deformable_groups)
        out = ops.mdcn_forward(_f32c(input), _f32c(offset), _f32c(mask), _f32c(weight),
                               _f32c(bias) if ctx.with_bias else None, stride, padding, dilation, groups,
                               deformable_groups)
        return out.to(input.dtype)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        if not grad_output.is_cuda:
            raise NotImplementedError
        input, offset, mask, weight, bias = ctx.saved_tensors
        if ctx.f64:
            gx, goff, gmask, gw, gb = _mdcn_backward_raw(_f64c(input), _f64c(offset), _f64c(mask), _f64c(weight),
                                                         _f64c(grad_output.double()), ctx.with_bias, ctx.stride,
                                                         ctx.padding, ctx.dilation, ctx.groups, ctx.deformable_groups)
            return gx, goff, gmask, gw, gb, None, None, None, None, None
        gx, goff, gmask, gw, gb = mdcn_backward(_f32c(input), _f32c(offset), _f32c(mask), _f32c(weight),
                                                _f32c(grad_output), ctx.with_bias, ctx.stride, ctx.padding,
                                                ctx.dilation, ctx.groups, ctx.deformable_groups)
        return (gx.to(input.dtype), goff.to(offset.dtype), gmask.to(mask.dtype), gw.to(weight.dtype),
                gb.to(bias.dtype) if ctx.with_bias else None, None, None, None, None, None)


def _pow2_scale(grad_out):
    """Device-side power of two s with amax(|grad_out| * s) in [2^9, 2^10): the backward kernels carry grad_out and
    W^T grad_out as fp16 tensor-core operands, so un-scaled gradients below ~6e-5 (mean-reduced losses, small loss weights,
    late training) would be subnormal or flush to zero and gradients above 65504 would overflow.  No host sync."""
    amax = grad_out.detach().abs().amax().clamp_min(1e-30).float()
    return torch.exp2(torch.floor(torch.log2(1024.0 / amax))).clamp(2.0 ** -100, 2.0 ** 100)


def mdcn_backward(x, offset, mask, weight, grad_out, with_bias, stride, padding, dilation, groups, dg):
    """All five gradients through eb_mdcn_backward (fp32 NCHW, reference layouts).  grad_out is pre-scaled by a power of two
    into the fp16 range of the kernels' operands and the (linear) results are scaled back - exact in fp32."""
    s = _pow2_scale(grad_out)
    grads = _mdcn_backward_raw(x, offset, mask, weight, (grad_out * s).contiguous(), with_bias, stride, padding, dilation,
                               groups, dg)
    inv = 1.0 / s
    return tuple(None if g is None else g * inv for g in grads)


def _mdcn_backward_raw(x, offset, mask, weight, grad_out, with_bias, stride, padding, dilation, groups, dg):
    N, C, H, W = x.shape
    Cout, _, kh, kw = weight.shape
    if groups > 1:          # composed from per-group calls (see ops.group_slices); shared deformable groups accumulate
        gx, gw = torch.empty_like(x), torch.empty_like(weight)
        goff, gmask = torch.zeros_like(offset), torch.zeros_like(mask)
        gb = torch.zeros(Cout, dtype=x.dtype, device=x.device) if with_bias else None
        for gi in range(groups):
            cs, os_, fs, ms, dgg = ops.group_slices(C, Cout, kh * kw, groups, dg, gi)
            r = _mdcn_backward_raw(x[:, cs].contiguous(), offset[:, fs].contiguous(), mask[:, ms].contiguous(),
                                   weight[os_].contiguous(), grad_out[:, os_].contiguous(), with_bias, stride, padding,
                                   dilation, 1, dgg)
            gx[:, cs], gw[os_] = r[0], r[3]
            goff[:, fs] += r[1]
            gmask[:, ms] += r[2]
            if with_bias:
                gb[os_] = r[4]
        return gx, goff, gmask, gw, gb
    gx = torch.empty_like(x)
    goff = torch.empty_like(offset)
    gmask = torch.empty_like(mask)
    gw = torch.zeros_like(weight)
    gb = torch.zeros(Cout, dtype=x.dtype, device=x.device) if with_bias else None
    if x.dtype == torch.float64:        # every tensor fp64: the double-precision kernels, no scaling needed
        need = L.lib().eb_mdcn_backward_f64_workspace(N, C, H, W, Cout, kh, kw, stride, padding, dilation)
        ws = torch.empty(max(need, 16), dtype=torch.uint8, device=x.device)
        L.check(L.lib().eb_mdcn_backward_f64(L.ptr(x), L.ptr(offset), L.ptr(mask), L.ptr(weight), L.ptr(grad_out),
                                             L.ptr(gx), L.ptr(goff), L.ptr(gmask), L.ptr(gw), L.ptr(gb), N, C, H, W, Cout,
                                             kh, kw, stride, padding, dilation, groups, dg, L.ptr(ws), ws.numel(),
                                             L.stream_ptr()), "eb_mdcn_backward_f64")
        return gx, goff, gmask, gw, gb
    need = L.lib().eb_mdcn_backward_workspace(N, C, H, W, Cout, kh, kw, stride, padding, dilation)
    ws = torch.empty(max(need, 16), dtype=torch.uint8, device=x.device)
    L.check(L.lib().eb_mdcn_backward(L.ptr(x), L.ptr(offset), L.ptr(mask), L.ptr(weight), L.ptr(grad_out),
                                     L.ptr(gx), L.ptr(goff), L.ptr(gmask), L.ptr(gw), L.ptr(gb), N, C, H, W, Cout,
                                     kh, kw, stride, padding, dilation, groups, dg, L.ptr(ws), ws.numel(),
                                     L.stream_ptr()), "eb_mdcn_backward")
    return gx, goff, gmask, gw, gb


modulated_deform_conv = ModulatedDeformConvFunction.apply


class DeformConvFunction(Function):
    """DCNv1 through the three eb_dcn1_* entry points (per-axis stride / padding / dilation)."""

    @staticmethod
    def forward(ctx, input, offset, weight, stride=1, padding=0, dilation=1, groups=1, deformable_groups=1,
                im2col_step=64):
        if input is not None and input.dim() != 4:
            raise ValueError(f"Expected 4D tensor as input, got {input.dim()}D tensor instead.")
        ctx.stride, ctx.padding, ctx.dilation = _pair(stride), _pair(padding), _pair(dilation)
        ctx.groups, ctx.deformable_groups, ctx.im2col_step = groups, deformable_groups, im2col_step
        ctx.save_for_backward(input, offset, weight)
        out_shape = DeformConvFunction._output_size(input, weight, ctx.padding, ctx.dilation, ctx.stride)
        if not input.is_cuda:
            raise NotImplementedError
        step = min(ctx.im2col_step, input.shape[0])
        assert (input.shape[0] % step) == 0, "im2col step must divide batchsize"
        ctx.f64 = _all_f64(input, offset, weight)
        cv = _f64c if ctx.f64 else _f32c
        output = torch.empty(out_shape, dtype=torch.float64 if ctx.f64 else torch.float32, device=input.device)
        from . import deform_conv_ext as ext
        ext.deform_conv_forward(cv(input), cv(weight), cv(offset), output, None, None, weight.size(3),
                                weight.size(2), ctx.stride[1], ctx.stride[0], ctx.padding[1], ctx.padding[0],
                                ctx.dilation[1], ctx.dilation[0], ctx.groups, ctx.deformable_groups, step)
        return output.to(input.dtype)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        input, offset, weight = ctx.saved_tensors
        grad_input = grad_offset = grad_weight = None
        if not grad_output.is_cuda:
            raise NotImplementedError
        step = min(ctx.im2col_step, input.shape[0])
        assert (input.shape[0] % step) == 0, "im2col step must divide batchsize"
        from . import deform_conv_ext as ext
        geom = (weight.size(3), weight.size(2), ctx.stride[1], ctx.stride[0], ctx.padding[1], ctx.padding[0],
                ctx.dilation[1], ctx.dilation[0], ctx.groups, ctx.deformable_groups)
        cv = (lambda t: _f64c(t.double())) if ctx.f64 else _f32c       # fp64 calls keep fp64 (grad_output included)
        x, off, go = cv(input), cv(offset), cv(grad_output)
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            gx, goff = torch.empty_like(x), torch.empty_like(off)
            ext.deform_conv_backward_input(x, off, go, gx, goff, cv(weight), None, *geom, step)
            grad_input, grad_offset = gx.to(input.dtype), goff.to(offset.dtype)
        if ctx.needs_input_grad[2]:
            gw = torch.zeros(weight.shape, dtype=x.dtype, device=weight.device)
            ext.deform_conv_backward_parameters(x, off, go, gw, None, None, *geom, 1, step)
            grad_weight = gw.to(weight.dtype)
        return grad_input, grad_offset, grad_weight, None, None, None, None, None, None

    @staticmethod
    def _output_size(input, weight, padding, dilation, stride):
        size = (input.size(0), weight.size(0))
        for d in range(input.dim() - 2):
            kernel = dilation[d] * (weight.size(d + 2) - 1) + 1
            size += ((input.size(d + 2) + 2 * padding[d] - kernel) // stride[d] + 1,)
        if not all(s > 0 for s in size):
            raise ValueError(f"convolution input is too small (output would be {'x'.join(map(str, size))})")
        return size


deform_conv = DeformConvFunction.apply


class ModulatedDeformConv(nn.Module):

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 deformable_groups=1, bias=True):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.kernel_size = _pair(kernel_size)
        self.stride = stride
        self.padding = padding
        self.dilation = dilation
        self.groups = groups
        self.deformable_groups = deformable_groups
        self.with_bias = bias
        self.transposed = False
        self.output_padding = _single(0)
        self.weight = nn.Parameter(torch.Tensor(out_channels, in_channels // groups, *self.kernel_size))
        if bias:
            self.bias = nn.Parameter(torch.Tensor(out_channels))
        else:
            self.register_parameter("bias", None)
        self.init_weights()

    def init_weights(self):
        n = self.in_channels
        for k in self.kernel_size:
            n *= k
        stdv = 1.0 / math.sqrt(n)
        self.weight.data.uniform_(-stdv, stdv)
        if self.bias is not None:
            self.bias.data.zero_()

    def forward(self, x, offset, mask):
        return modulated_deform_conv(x, offset, mask, self.weight, self.bias, self.stride, self.padding,
                                     self.dilation, self.groups, self.deformable_groups)


class ModulatedDeformConvPack(ModulatedDeformConv):
    """conv_offset (zero-initialised) + modulated deformable conv, like the reference's Pack."""

    _version = 2

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.conv_offset = nn.Conv2d(self.in_channels,
                                     self.deformable_groups * 3 * self.kernel_size[0] * self.kernel_size[1],
                                     kernel_size=self.kernel_size, stride=_pair(self.stride),
                                     padding=_pair(self.padding), dilation=_pair(self.dilation), bias=True)
        self.init_weights()
        self._packed = None

    def init_weights(self):
        super().init_weights()
        if hasattr(self, "conv_offset"):
            self.conv_offset.weight.data.zero_()
            self.conv_offset.bias.data.zero_()

    # -- fused inference path: conv_offset -> packed (offset, sigmoid(mask)) -> DCN, no host sync
    def _fusable(self, x):
        k = self.kernel_size
        return (not torch.is_grad_enabled() and x.is_cuda and k == (3, 3) and self.stride == 1 and self.padding == 1
                and not (x.dtype == torch.float64 and self.weight.dtype == torch.float64)   # fp64 module: fp64 operator
                and self.dilation == 1 and self.groups == 1 and self.in_channels % 64 == 0
                and ((self.in_channels // self.deformable_groups) == 8 or (self.in_channels // self.deformable_groups) % 16 == 0))

    def _site(self):
        key = tuple(int(p._version) for p in self.parameters()) + (self.weight.data_ptr(),)
        if self._packed is None or self._packed[0] != key:
            site = ops.DcnSite(self.conv_offset.weight.detach().float(), self.conv_offset.bias.detach().float(),
                               self.weight.detach().float(), None if self.bias is None else self.bias.detach().float(),
                               self.deformable_groups)
            self._packed = (key, site)
        return self._packed[1]

    def _fused_forward(self, x, feat):
        """One launch (dcn_site.cuh): conv_offset on the tensor cores, offsets and masks stay in tensor memory; the
        reference's `offset_absmean > 50` warning is accumulated on the device and reported by the next call."""
        _MONITOR.poll()
        site = self._site()
        with torch.cuda.device(x.device):
            xv, fv = ops.nchw_to_nhwc(x.float()), ops.nchw_to_nhwc(feat.float())
            acc = torch.zeros(1, dtype=torch.float32, device=x.device)
            out = torch.empty(xv.N, self.out_channels, xv.H, xv.W, dtype=torch.float32, device=x.device)
            site(xv, fv, absmean=acc, out_nchw=out)
            n = fv.N * fv.H * fv.W * self.deformable_groups * 18
            self.last_offset_abssum = (acc, n)
            _MONITOR.submit(acc, [n])
        return out.to(x.dtype)

    def forward(self, x):
        if self._fusable(x):
            return self._fused_forward(x, x)
        out = self.conv_offset(x)
        o1, o2, mask = torch.chunk(out, 3, dim=1)
        offset = torch.cat((o1, o2), dim=1)
        mask = torch.sigmoid(mask)
        return modulated_deform_conv(x, offset, mask, self.weight, self.bias, self.stride, self.padding,
                                     self.dilation, self.groups, self.deformable_groups)


class DCNv2Pack(ModulatedDeformConvPack):
    """Offsets and masks come from a second feature map (arch_util.py:232-257).

    The reference's `offset_absmean > 50` warning forces a device->host sync on every call (arch_util.py:249-253).  On the
    fused inference path the sum is accumulated on the device and the warning is emitted by the NEXT DCN call once the
    asynchronous read-back has finished (ops.OffsetMonitor); ``check_offset_absmean()`` forces it for the last call.  Under
    autograd (training) the reference's immediate check is kept.
    """

    def forward(self, x, feat):
        if self._fusable(x):
            return self._fused_forward(x, feat)
        out = self.conv_offset(feat)
        o1, o2, mask = torch.chunk(out, 3, dim=1)
        offset = torch.cat((o1, o2), dim=1)
        mask = torch.sigmoid(mask)
        offset_absmean = torch.mean(torch.abs(offset.detach()))
        self.last_offset_abssum = (offset.detach().abs().sum().reshape(1), offset.numel())
        if offset_absmean > 50:          # arch_util.py:249-253 (the training-divergence signal): immediate, like the reference
            logging.getLogger("basicsr").warning(f"Offset abs mean is {offset_absmean}, larger than 50.")
        return modulated_deform_conv(x, offset, mask, self.weight, self.bias, self.stride, self.padding,
                                     self.dilation, self.groups, self.deformable_groups)

    def check_offset_absmean(self):
        acc, n = getattr(self, "last_offset_abssum", (None, 0))
        if acc is None:
            return None
        mean = float(acc.item()) / max(n, 1)
        if mean > 50:
            logging.getLogger("basicsr").warning(f"Offset abs mean is {mean}, larger than 50.")
        return mean


class DeformConv(nn.Module):
    """DCNv1 layer with external offsets; parameters and init as deform_conv.py:186-247 (bias is not supported there)."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 deformable_groups=1, bias=False):
        super().__init__()
        assert not bias
        assert in_channels % groups == 0, f"in_channels {in_channels} is not divisible by groups {groups}"
        assert out_channels % groups == 0, f"out_channels {out_channels} is not divisible by groups {groups}"
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride = _pair(kernel_size), _pair(stride)
        self.padding, self.dilation = _pair(padding), _pair(dilation)
        self.groups, self.deformable_groups = groups, deformable_groups
        self.transposed, self.output_padding = False, _single(0)     # nn.Conv2d look-alike attributes
        self.weight = nn.Parameter(torch.Tensor(out_channels, in_channels // groups, *self.kernel_size))
        self.reset_parameters()

    def reset_parameters(self):
        stdv = 1.0 / math.sqrt(self.in_channels * self.kernel_size[0] * self.kernel_size[1])
        self.weight.data.uniform_(-stdv, stdv)

    def forward(self, x, offset):
        # inputs smaller than the kernel are zero-padded on the bottom/right and the output cropped back
        # (deform_conv.py:232-247)
        pad_h = max(self.kernel_size[0] - x.size(2), 0)
        pad_w = max(self.kernel_size[1] - x.size(3), 0)
        if pad_h or pad_w:
            x = nn.functional.pad(x, (0, pad_w, 0, pad_h), "constant", 0).contiguous()
            offset = nn.functional.pad(offset, (0, pad_w, 0, pad_h), "constant", 0).contiguous()
        out = deform_conv(x, offset, self.weight, self.stride, self.padding, self.dilation, self.groups,
                          self.deformable_groups)
        if pad_h or pad_w:
            out = out[:, :, :out.size(2) - pad_h, :out.size(3) - pad_w].contiguous()
        return out


class DeformConvPack(DeformConv):
    """DCNv1 layer that predicts its own offsets with a zero-initialised conv (deform_conv.py:250-292)."""

    _version = 2

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.conv_offset = nn.Conv2d(self.in_channels,
                                     self.deformable_groups * 2 * self.kernel_size[0] * self.kernel_size[1],
                                     kernel_size=self.kernel_size, stride=_pair(self.stride),
                                     padding=_pair(self.padding), dilation=_pair(self.dilation), bias=True)
        self.init_offset()

    def init_offset(self):
        self.conv_offset.weight.data.zero_()
        self.conv_offset.bias.data.zero_()

    def forward(self, x):
        offset = self.conv_offset(x)
        return deform_conv(x, offset, self.weight, self.stride, self.padding, self.dilation, self.groups,
                           self.deformable_groups)


__all__ = ["DeformConv", "DeformConvPack", "ModulatedDeformConv", "ModulatedDeformConvPack", "deform_conv",
           "modulated_deform_conv", "DCNv2Pack"]
