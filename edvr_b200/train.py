"""Training step of EDVR on the B200 kernels (BASELINE cfg 5: EDVR-L 4x SR, bf16, Charbonnier loss, DCNv2 backward, DDP).

What the reference does for a step (basicsr/models/edvr_model.py + sr_model.py optimize_parameters, net wrapped in
DistributedDataParallel at base_model.py:62-69, options/train/EDVR/train_EDVR_L_x4_SR_REDS.yml): the fp32 graph of
edvr_arch.py under autograd - cuDNN forward / dgrad / wgrad for ~100 convolutions, the dcn extension's forward / backward
for 4 sites x t frames - then Adam and NCCL all-reduce of 82.5 MB of gradients.

Here every convolution of that graph is ONE autograd Function on NHWC 16-bit activations (bf16 by default, the dtype cfg 5
names; fp16 selectable):
  forward  : conv_pair_kernel (CTA-pair tcgen05 implicit GEMM, TMA in/out), bias + ReLU/LeakyReLU fused
  dgrad    : the same kernel on the transposed, spatially flipped weights (a stride-1 conv of grad_out)
  wgrad    : conv_wgrad_kernel (conv_train.cuh): split-K tcgen05 GEMM over channel-major transposes of x and grad_out
  stride 2 : computed at stride 1 and sampled at even pixels (as the inference executor does); backward zero-stuffs
and the DCN sites run edvr_b200.dcn.modulated_deform_conv (our fused forward + backward kernels, fp32 operator boundary).
The elementwise glue (activations' derivatives, cat, bilinear resize, pooling, pixel shuffle, the TSA products, the loss) is
plain PyTorch on the same NHWC tensors - no cuDNN kernel runs in a step.  Parameters, gradients and the optimizer state stay
fp32 (master weights); weights are re-packed into the MMA layout on every call because they change every step.
"""
import ctypes

import torch
import torch.nn.functional as F
from torch.autograd import Function

from . import _lib as L
from . import ops
from .dcn import modulated_deform_conv
from .ops import ACT_LRELU, ACT_NONE, ACT_RELU, PackedConv, View

_WS = {}


def _workspace(nbytes, device):
    """One growing scratch buffer per device for the wgrad transposes (stream-ordered reuse)."""
    t = _WS.get(device)
    if t is None or t.numel() < nbytes:
        t = _WS[device] = torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=device)
    return t


def _pack_pair(weight, bias, bf16, dgrad_k=0):
    """fp32 master weights [Cout, Cin, k, k] -> PackedConv for the CTA-pair kernel only (no single-CTA copy).
    dgrad_k == 0: the forward convolution (Cin % 64 == 0).  dgrad_k > 0: the DATA-GRADIENT convolution, i.e. weights
    W'[ci][co][flipped tap] with `dgrad_k` (>= Cout, multiple of 64) grad_out channels, packed straight from `weight`."""
    weight = weight.detach()
    if weight.dtype != torch.float32 or not weight.is_contiguous():
        weight = weight.float().contiguous()
    cout, cin, k, _ = weight.shape
    rows, kch = (cout, cin) if not dgrad_k else (cin, dgrad_k)
    cp = ((rows + 31) // 32) * 32
    pc = PackedConv()
    pc.BN = ops._choose_bn(cp)
    pc.n_tiles = cp // pc.BN
    pc.cin, pc.ksize, pc.cout, pc.cin_real = kch, k, rows, kch
    if not L.lib().eb_conv2d_pair_supported(kch, k, pc.BN, pc.n_tiles):
        raise ValueError(f"conv {kch}->{rows} k{k}: outside the CTA-pair kernel (Cin % 64 == 0, k in (1, 3))")
    nbytes = L.lib().eb_packed_weight_bytes(kch, k * k, pc.BN, pc.n_tiles)
    pc.w = None
    pc.wpair = torch.empty(nbytes // 2, dtype=torch.float16, device=weight.device)      # raw 16-bit storage
    with ops._Rec("pack_weight", 1):
        if dgrad_k:
            L.check(L.lib().eb_pack_weight_pair_dgrad(L.ptr(weight), cout, cin, k * k, kch, pc.BN, pc.n_tiles, L.ptr(pc.wpair),
                                                      1 if bf16 else 0, L.stream_ptr()), "eb_pack_weight_pair_dgrad")
        else:
            L.check(L.lib().eb_pack_weight_pair_ex(L.ptr(weight), cout, cin, k * k, pc.BN, pc.n_tiles, L.ptr(pc.wpair),
                                                   1 if bf16 else 0, L.stream_ptr()), "eb_pack_weight_pair_ex")
    if bias is not None and cp == rows and bias.dtype == torch.float32 and bias.is_contiguous():
        pc.b = bias.detach()
    elif bias is not None:
        pc.b = torch.zeros(cp, dtype=torch.float32, device=weight.device)
        pc.b[:rows] = bias.detach().float()
    else:
        pc.b = None
    return pc


def _pad_channels(t, mult=64):
    """[N,H,W,C] -> [N,H,W,ceil(C/mult)*mult] with zero channels appended (Cin of the tensor-core kernels)."""
    c = t.shape[3]
    cp = ((c + mult - 1) // mult) * mult
    if cp == c:
        return t
    out = t.new_zeros(t.shape[0], t.shape[1], t.shape[2], cp)
    out[..., :c] = t
    return out


def _run_conv(x, weight, bias, act, dgrad=False):
    """y = act(conv(x) + bias); x NHWC 16-bit contiguous with C % 64 == 0 -> y NHWC (same dtype).  dgrad: x is grad_out
    (channels padded to 64) and the result is the gradient w.r.t. the convolution's input, [N,H,W,Cin]."""
    bf16 = x.dtype == torch.bfloat16
    pc = _pack_pair(weight, bias, bf16, dgrad_k=x.shape[3] if dgrad else 0)
    N, H, W, _ = x.shape
    cp = pc.BN * pc.n_tiles
    y = torch.empty(N, H, W, cp, dtype=x.dtype, device=x.device)
    ops.conv2d(pc, [View(x)], out16=View(y), act=act)
    return y if cp == pc.cout else y[..., :pc.cout].contiguous()


class _ConvFn(Function):
    """3x3 (pad 1) / 1x1 convolution, stride 1 or 2, on NHWC 16-bit activations with fp32 master weights."""

    @staticmethod
    def forward(ctx, x, weight, bias, act, stride):
        x = x.contiguous()
        cin_real = x.shape[3]
        xp = _pad_channels(x)
        w = weight if xp.shape[3] == cin_real else F.pad(weight, (0, 0, 0, 0, 0, xp.shape[3] - cin_real))
        with torch.cuda.device(x.device):
            y = _run_conv(xp, w, bias, act)
        if stride == 2:
            y = y[:, ::2, ::2].contiguous()          # k3/s2/p1 == the stride-1 result at even pixels
        ctx.save_for_backward(xp, weight, y if act != ACT_NONE else None)
        ctx.act, ctx.stride, ctx.cin_real, ctx.has_bias = act, stride, cin_real, bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        xp, weight, y = ctx.saved_tensors
        act, stride, cin_real = ctx.act, ctx.stride, ctx.cin_real
        bf16 = xp.dtype == torch.bfloat16
        gy = gy.contiguous()
        if act == ACT_RELU:
            gy = torch.ops.aten.threshold_backward(gy, y, 0)                  # one elementwise pass on the saved output
        elif act == ACT_LRELU:
            gy = torch.ops.aten.leaky_relu_backward(gy, y, 0.1, True)
        N, H, W, cin = xp.shape
        cout, _, k, _ = weight.shape
        if stride == 2:                                # zero-stuff to the stride-1 grid
            full = gy.new_zeros(N, H, W, cout)
            full[:, ::2, ::2] = gy
            gy = full
        gx = gw = gb = None
        with torch.cuda.device(xp.device):
            if ctx.needs_input_grad[0]:
                # dgrad: conv of grad_out with W'[ci][co][ky][kx] = W[co][ci][2-ky][2-kx]; grad_out channels padded to 64
                gx = _run_conv(_pad_channels(gy), weight, None, ACT_NONE, dgrad=True)      # [N,H,W,cin_real]
            if ctx.needs_input_grad[1]:
                want_gb = ctx.has_bias and ctx.needs_input_grad[2]
                # one zero-filled fp32 buffer for grad_weight (+ grad_bias): the kernels accumulate into it
                buf = torch.zeros(cout * cin * k * k + (cout if want_gb else 0), dtype=torch.float32, device=xp.device)
                gwp = buf[:cout * cin * k * k].view(cout, cin, k, k)
                gb = buf[cout * cin * k * k:] if want_gb else None
                need = L.lib().eb_conv_wgrad_workspace(N, H, W, cin, cout, k)
                ws = _workspace(need, xp.device)
                with ops._Rec("conv_wgrad", 4, 2.0 * N * H * W * cout * cin * k * k):
                    L.check(L.lib().eb_conv_wgrad(L.ptr(xp), cin, 0, L.ptr(gy), cout, 0, N, H, W, cin, cout, k,
                                                  1 if bf16 else 0, 1.0, L.ptr(gwp), L.ptr(gb), L.ptr(ws), ws.numel(),
                                                  L.stream_ptr()), "eb_conv_wgrad")
                gw = gwp if cin == cin_real else gwp[:, :cin_real].contiguous()
            elif ctx.has_bias and ctx.needs_input_grad[2]:
                gb = gy.sum((0, 1, 2), dtype=torch.float32)
        return gx, gw, gb, None, None


def conv(x, m, act=ACT_NONE):
    """nn.Conv2d module `m` (3x3 pad 1 or 1x1, stride 1 or 2) applied to the NHWC 16-bit tensor x on the tensor-core kernels."""
    return _ConvFn.apply(x, m.weight, m.bias, act, m.stride[0])


def _nchw(t):           # NHWC tensor -> its NCHW view (channels_last memory format: no copy)
    return t.permute(0, 3, 1, 2)


def _nhwc(t):           # NCHW view in channels_last -> NHWC tensor (no copy when already channels_last)
    return t.permute(0, 2, 3, 1).contiguous()


def up2(t):
    return _nhwc(F.interpolate(_nchw(t), scale_factor=2, mode="bilinear", align_corners=False))


def dcn_pack(m, x, feat):
    """DCNv2Pack.forward (arch_util.py:243-257) under autograd: conv_offset on the conv Function, the deformable conv on
    edvr_b200.dcn.modulated_deform_conv (fused forward kernel + backward kernels, fp32 NCHW operator boundary)."""
    import logging
    out = _nchw(conv(feat, m.conv_offset)).float()
    o1, o2, mask = torch.chunk(out, 3, dim=1)
    offset = torch.cat((o1, o2), dim=1)
    mask = torch.sigmoid(mask)
    if not torch.cuda.is_current_stream_capturing():
        # the reference's immediate check (arch_util.py:249-253, the training-divergence signal); it is a device->host sync,
        # so it is left out of a CUDA-graph capture of the step (GraphedTrainStep) - replay cannot branch on the host
        offset_absmean = torch.mean(torch.abs(offset.detach()))
        if offset_absmean > 50:
            logging.getLogger("basicsr").warning(f"Offset abs mean is {offset_absmean}, larger than 50.")
    y = modulated_deform_conv(_nchw(x).float().contiguous(), offset.contiguous(), mask.contiguous(), m.weight, m.bias,
                              m.stride, m.padding, m.dilation, m.groups, m.deformable_groups)
    return _nhwc(y.to(x.dtype))


def resblock(m, x):
    return x + conv(conv(x, m.conv1, ACT_RELU), m.conv2)


def pcd_align(m, nbr, ref):
    """PCDAlignment.forward (edvr_arch.py:76-117) on NHWC tensors."""
    up_off = up_feat = feat = None
    for i in (3, 2, 1):
        Lv = f"l{i}"
        off = conv(torch.cat([nbr[i - 1], ref[i - 1]], 3), m.offset_conv1[Lv], ACT_LRELU)
        if i == 3:
            off = conv(off, m.offset_conv2[Lv], ACT_LRELU)
        else:
            off = conv(conv(torch.cat([off, up_off], 3), m.offset_conv2[Lv], ACT_LRELU), m.offset_conv3[Lv], ACT_LRELU)
        feat = dcn_pack(m.dcn_pack[Lv], nbr[i - 1], off)
        if i < 3:
            feat = conv(torch.cat([feat, up_feat], 3), m.feat_conv[Lv])
        if i > 1:
            feat = F.leaky_relu(feat, 0.1)
            up_off, up_feat = up2(off) * 2, up2(feat)
    off = conv(conv(torch.cat([feat, ref[0]], 3), m.cas_offset_conv1, ACT_LRELU), m.cas_offset_conv2, ACT_LRELU)
    return F.leaky_relu(dcn_pack(m.cas_dcnpack, feat, off), 0.1)


def tsa_fusion(m, aligned):
    """TSAFusion.forward (edvr_arch.py:161-214); aligned: [b, t, h, w, c]."""
    b, t, h, w, c = aligned.shape
    emb_ref = conv(aligned[:, m.center_frame_idx].contiguous(), m.temporal_attn1)
    emb = conv(aligned.reshape(b * t, h, w, c), m.temporal_attn2).view(b, t, h, w, c)
    prob = torch.sigmoid((emb.float() * emb_ref.float().unsqueeze(1)).sum(4, keepdim=True)).to(aligned.dtype)
    x = (aligned * prob).permute(0, 2, 3, 1, 4).reshape(b, h, w, t * c)           # channel index = frame * c + ch
    feat = conv(x, m.feat_fusion, ACT_LRELU)
    attn = conv(x, m.spatial_attn1, ACT_LRELU)

    def pools(z):
        zc = _nchw(z)
        return torch.cat([_nhwc(F.max_pool2d(zc, 3, 2, 1)), _nhwc(F.avg_pool2d(zc, 3, 2, 1))], 3)

    attn = conv(pools(attn), m.spatial_attn2, ACT_LRELU)
    lvl = conv(attn, m.spatial_attn_l1, ACT_LRELU)
    lvl = conv(pools(lvl), m.spatial_attn_l2, ACT_LRELU)
    lvl = up2(conv(lvl, m.spatial_attn_l3, ACT_LRELU))
    attn = up2(conv(conv(attn, m.spatial_attn3, ACT_LRELU) + lvl, m.spatial_attn4, ACT_LRELU))
    attn = conv(attn, m.spatial_attn5)
    add = conv(conv(attn, m.spatial_attn_add1, ACT_LRELU), m.spatial_attn_add2)
    return feat * torch.sigmoid(attn) * 2 + add


def predeblur(m, x):
    """PredeblurModule.forward (edvr_arch.py:250-269)."""
    l1 = conv(x, m.conv_first, ACT_LRELU)
    if m.hr_in:
        l1 = conv(conv(l1, m.stride_conv_hr1, ACT_LRELU), m.stride_conv_hr2, ACT_LRELU)
    l2 = conv(l1, m.stride_conv_l2, ACT_LRELU)
    l3 = conv(l2, m.stride_conv_l3, ACT_LRELU)
    l3 = up2(resblock(m.resblock_l3, l3))
    l2 = up2(resblock(m.resblock_l2_2, resblock(m.resblock_l2_1, l2) + l3))
    for i in range(2):
        l1 = resblock(m.resblock_l1[i], l1)
    l1 = l1 + l2
    for i in range(2, 5):
        l1 = resblock(m.resblock_l1[i], l1)
    return l1


def edvr_forward(net, x, dtype=torch.bfloat16):
    """EDVR.forward (edvr_arch.py:358-420) as a differentiable graph on the B200 kernels.  x: fp32 [b, t, 3, h, w] (CUDA);
    returns fp32 [b, 3, 4h, 4w] ([b, 3, h, w] with hr_in)."""
    b, t, c, h, w = x.shape
    xc = x[:, net.center_frame_idx].contiguous()
    frames = x.reshape(b * t, c, h, w).permute(0, 2, 3, 1).to(dtype).contiguous()            # NHWC
    if net.with_predeblur:
        l1 = conv(predeblur(net.predeblur, frames), net.conv_1x1)
        if net.hr_in:
            h, w = h // 4, w // 4
    else:
        l1 = conv(frames, net.conv_first, ACT_LRELU)
    for blk in net.feature_extraction:
        l1 = resblock(blk, l1)
    l2 = conv(conv(l1, net.conv_l2_1, ACT_LRELU), net.conv_l2_2, ACT_LRELU)
    l3 = conv(conv(l2, net.conv_l3_1, ACT_LRELU), net.conv_l3_2, ACT_LRELU)
    C = l1.shape[3]
    l1, l2, l3 = l1.view(b, t, h, w, C), l2.view(b, t, h // 2, w // 2, C), l3.view(b, t, h // 4, w // 4, C)
    ci = net.center_frame_idx
    # all t neighbour frames of all clips go through PCD alignment as ONE batch (the reference loops over frames in Python,
    # edvr_arch.py:397-402; samples are independent, so the result is the same): reference features repeated per frame
    def rep(z):
        return z[:, ci].unsqueeze(1).expand(-1, t, -1, -1, -1).reshape(b * t, *z.shape[2:])
    nbr = [z.reshape(b * t, *z.shape[2:]) for z in (l1, l2, l3)]
    aligned = pcd_align(net.pcd_align, nbr, [rep(l1), rep(l2), rep(l3)]).view(b, t, h, w, C)
    if net.with_tsa:
        feat = tsa_fusion(net.fusion, aligned)
    else:
        feat = conv(aligned.permute(0, 2, 3, 1, 4).reshape(b, h, w, t * C), net.fusion)
    out = feat
    for blk in net.reconstruction:
        out = resblock(blk, out)
    out = F.leaky_relu(_nhwc(F.pixel_shuffle(_nchw(conv(out, net.upconv1)), 2)), 0.1)
    out = F.leaky_relu(_nhwc(F.pixel_shuffle(_nchw(conv(out, net.upconv2)), 2)), 0.1)
    out = conv(conv(out, net.conv_hr, ACT_LRELU), net.conv_last)
    out = _nchw(out).float()
    base = xc if net.hr_in else F.interpolate(xc, scale_factor=4, mode="bilinear", align_corners=False)
    return out + base


def charbonnier_loss(pred, target, eps=1e-12, reduction="sum", loss_weight=1.0):
    """basicsr/models/losses/losses.py:24-25,115-150 (CharbonnierLoss; the REDS yml uses reduction='sum')."""
    v = torch.sqrt((pred - target) ** 2 + eps)
    return loss_weight * (v.sum() if reduction == "sum" else v.mean())


class GraphedTrainStep:
    """One optimisation step (forward, loss, backward, optimizer.step) captured ONCE into a CUDA graph and replayed:
    an EDVR-L step is ~4000 small launches (weight packs, transposes, elementwise glue, 20 DCN calls) and is host-bound when
    issued eagerly; every shape is static, so the whole step replays from one launch.  The optimizer must be capturable
    (torch.optim.Adam(..., capturable=True)).  __call__(x, target) copies the batch into the static buffers, replays,
    and returns the (static) loss tensor."""

    def __init__(self, net, optimizer, loss_fn, x, target, warmup=3):
        self.x, self.target = x.clone(), target.clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):                       # allocate workspaces / optimizer state outside the capture
                optimizer.zero_grad(set_to_none=True)
                loss_fn(net(self.x), self.target).backward()
                optimizer.step()
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            optimizer.zero_grad(set_to_none=True)
            with torch.cuda.graph(self.graph, stream=side):
                self.loss = loss_fn(net(self.x), self.target)
                self.loss.backward()
                optimizer.step()
        torch.cuda.current_stream().wait_stream(side)

    def __call__(self, x=None, target=None):
        if x is not None:
            self.x.copy_(x, non_blocking=True)
        if target is not None:
            self.target.copy_(target, non_blocking=True)
        self.graph.replay()
        return self.loss
