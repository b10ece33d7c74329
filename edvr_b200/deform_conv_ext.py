"""B1 boundary: a drop-in for the compiled module ``basicsr.models.ops.dcn.deform_conv_ext``.

Exposes all five pybind11 names (DCNv2 forward/backward, DCNv1 forward/backward_input/backward_parameters) of /root/reference/basicsr/models/ops/dcn/src/deform_conv_ext.cpp:149-163 with the
same positional signatures and in-place ownership rules (caller allocates every output; grad_weight / grad_bias are
accumulated into; `ones` / `columns` are legacy scratch handles and are ignored), implemented over the C ABI of
libedvr_b200.so.  Register it BEFORE importing basicsr and the unmodified reference tree runs on the B200 kernels:

    import sys, edvr_b200.deform_conv_ext as ext
    sys.modules["basicsr.models.ops.dcn.deform_conv_ext"] = ext

Errors surface as RuntimeError with the library's message (the reference raises through TORCH_CHECK / AT_ERROR);
CPU tensors raise RuntimeError("... not implemented on CPU") like deform_conv_ext.cpp:123,145.
"""
import torch

from . import _lib as L


def _check_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(f"{what} is not implemented on CPU")


def _f32(t):
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()


def _all_f64(*ts):
    """True when every floating tensor of a call (None = absent) is float64: such calls run the double-precision entry
    points as given - no cast and no grad_out scaling."""
    return all(t is None or t.dtype == torch.float64 for t in ts)


def _pow2_scale(grad_out):
    """Power of two s (computed on the device, no host sync) with amax(|grad_out|) * s in [2^9, 2^10): the backward kernels
    carry grad_out and W^T grad_out as fp16 tensor-core operands, so gradients of a mean-reduced loss (~1e-6 per pixel)
    would be subnormal or flush to zero un-scaled, and very large ones overflow at 65504.  All results are linear in
    grad_out, so dividing them by s afterwards is exact."""
    amax = grad_out.detach().abs().amax().clamp_min(1e-30).float()
    return torch.exp2(torch.floor(torch.log2(1024.0 / amax))).clamp(2.0 ** -100, 2.0 ** 100)


def modulated_deform_conv_forward(input, weight, bias, ones, offset, mask, output, columns, kernel_h, kernel_w,
                                  stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group, deformable_group,
                                  with_bias):
    _check_cuda(input, "modulated deform conv")
    if not input.is_contiguous():
        raise RuntimeError("input tensor has to be contiguous")      # deform_conv_cuda.cpp:497
    if not weight.is_contiguous():
        raise RuntimeError("weight tensor has to be contiguous")     # deform_conv_cuda.cpp:498
    if (stride_h, pad_h, dilation_h) != (stride_w, pad_w, dilation_w):
        raise RuntimeError("edvr_b200: anisotropic stride/pad/dilation is not supported (the v2 Python API passes one int)")
    if tuple(weight.shape[2:]) != (kernel_h, kernel_w):
        raise RuntimeError(f"Input shape and kernel shape wont match: ({kernel_h} x {kernel_w} vs "
                           f"{weight.shape[2]} x {weight.shape[3]}).")
    N, C, H, W = input.shape
    Cout = weight.shape[0]
    if C != weight.shape[1] * group:
        raise RuntimeError(f"Input shape and kernel channels wont match: ({C} vs {weight.shape[1] * group}).")
    halves = [input, weight, offset, mask, output] + ([bias] if with_bias else [])
    if group == 1 and all(t.dtype == torch.float16 and t.is_contiguous() for t in halves):
        # at::Half tensors (the reference dispatches on them: deform_conv_cuda_kernel.cu:781): the fp16 entry point, no casts
        need = L.lib().eb_mdcn_forward_f16_workspace(N, C, H, W, Cout, kernel_h, kernel_w, deformable_group)
        ws = torch.empty(max(need, 16), dtype=torch.uint8, device=input.device)
        with torch.cuda.device(input.device):
            L.check(L.lib().eb_mdcn_forward_f16(L.ptr(input), L.ptr(offset), L.ptr(mask), L.ptr(weight),
                                                L.ptr(bias if with_bias else None), L.ptr(output), N, C, H, W, Cout, kernel_h,
                                                kernel_w, stride_h, pad_h, dilation_h, group, deformable_group, L.ptr(ws),
                                                ws.numel(), L.stream_ptr()), "eb_mdcn_forward_f16")
        return
    if _all_f64(input, weight, offset, mask, output, bias if with_bias else None):
        from . import ops          # groups > 1: the per-group composition of ops.mdcn_forward, each call fp64
        with torch.cuda.device(input.device):
            output.copy_(ops.mdcn_forward(input, offset.contiguous(), mask.contiguous(), weight,
                                          bias.contiguous() if with_bias else None, stride_h, pad_h, dilation_h, group,
                                          deformable_group))
        return
    x, w, off, m = _f32(input), _f32(weight), _f32(offset), _f32(mask)
    b = _f32(bias) if with_bias else None
    if group > 1:           # deform_conv_cuda.cpp:536-568: one GEMM per weight group; composed from per-group calls
        from . import ops
        with torch.cuda.device(input.device):
            output.copy_(ops.mdcn_forward(x, off, m, w, b, stride_h, pad_h, dilation_h, group, deformable_group))
        return
    out32 = output if (output.dtype == torch.float32 and output.is_contiguous()) else torch.empty(
        output.shape, dtype=torch.float32, device=output.device)
    need = L.lib().eb_mdcn_forward_workspace(N, C, H, W, Cout, kernel_h, kernel_w)
    ws = torch.empty(max(need, 16), dtype=torch.uint8, device=input.device)
    with torch.cuda.device(input.device):                           # at::DeviceGuard, deform_conv_cuda.cpp:499
        L.check(L.lib().eb_mdcn_forward(L.ptr(x), L.ptr(off), L.ptr(m), L.ptr(w), L.ptr(b), L.ptr(out32), N, C, H, W,
                                        Cout, kernel_h, kernel_w, stride_h, pad_h, dilation_h, group, deformable_group,
                                        L.ptr(ws), ws.numel(), L.stream_ptr()), "eb_mdcn_forward")
    if out32 is not output:
        output.copy_(out32)


def modulated_deform_conv_backward(input, weight, bias, ones, offset, mask, columns, grad_input, grad_weight,
                                   grad_bias, grad_offset, grad_mask, grad_output, kernel_h, kernel_w, stride_h,
                                   stride_w, pad_h, pad_w, dilation_h, dilation_w, group, deformable_group, with_bias):
    _check_cuda(input, "modulated deform conv")
    if not input.is_contiguous():
        raise RuntimeError("input tensor has to be contiguous")
    if not weight.is_contiguous():
        raise RuntimeError("weight tensor has to be contiguous")
    if (stride_h, pad_h, dilation_h) != (stride_w, pad_w, dilation_w):
        raise RuntimeError("edvr_b200: anisotropic stride/pad/dilation is not supported")
    N, C, H, W = input.shape
    Cout = weight.shape[0]
    if _all_f64(input, weight, offset, mask, grad_input, grad_weight, grad_offset, grad_mask, grad_output,
                *((bias, grad_bias) if with_bias else ())):
        from .dcn import _mdcn_backward_raw       # groups > 1: its per-group composition, each call fp64
        with torch.cuda.device(input.device):
            gx, goff, gm, gw, gb = _mdcn_backward_raw(input, offset.contiguous(), mask.contiguous(), weight,
                                                      grad_output.contiguous(), bool(with_bias), stride_h, pad_h,
                                                      dilation_h, group, deformable_group)
        grad_input.copy_(gx)
        grad_offset.copy_(goff)
        grad_mask.copy_(gm)
        grad_weight.add_(gw)
        if with_bias:
            grad_bias.add_(gb)
        return
    x, w, off, m = _f32(input), _f32(weight), _f32(offset), _f32(mask)
    sc = _pow2_scale(grad_output)
    go = (grad_output.float() * sc).contiguous()
    inv = 1.0 / sc
    new = lambda t: torch.empty(t.shape, dtype=torch.float32, device=t.device)
    if group > 1:           # deform_conv_cuda.cpp:617-671 per weight group; composed from per-group calls
        from .dcn import _mdcn_backward_raw
        with torch.cuda.device(input.device):
            gx, goff, gm, gw, gb = _mdcn_backward_raw(x, off, m, w, go, bool(with_bias), stride_h, pad_h, dilation_h, group,
                                                      deformable_group)
    else:
        gx, goff, gm = new(grad_input), new(grad_offset), new(grad_mask)
        gw = torch.zeros(grad_weight.shape, dtype=torch.float32, device=grad_weight.device)
        gb = torch.zeros(grad_bias.shape, dtype=torch.float32, device=grad_bias.device) if with_bias else None
        need = L.lib().eb_mdcn_backward_workspace(N, C, H, W, Cout, kernel_h, kernel_w, stride_h, pad_h, dilation_h)
        ws = torch.empty(max(need, 16), dtype=torch.uint8, device=input.device)
        with torch.cuda.device(input.device):
            L.check(L.lib().eb_mdcn_backward(L.ptr(x), L.ptr(off), L.ptr(m), L.ptr(w), L.ptr(go), L.ptr(gx), L.ptr(goff),
                                             L.ptr(gm), L.ptr(gw), L.ptr(gb), N, C, H, W, Cout, kernel_h, kernel_w,
                                             stride_h, pad_h, dilation_h, group, deformable_group, L.ptr(ws), ws.numel(),
                                             L.stream_ptr()), "eb_mdcn_backward")
    grad_input.copy_(gx * inv)                  # overwritten, like deform_conv_cuda.cpp:617-657
    grad_offset.copy_(goff * inv)
    grad_mask.copy_(gm * inv)
    grad_weight.add_((gw * inv).to(grad_weight.dtype))        # accumulated into, like deform_conv_cuda.cpp:659-671
    if with_bias:
        grad_bias.add_((gb * inv).to(grad_bias.dtype))


def _v1_shape_check(input, offset, grad_output, weight, kH, kW, dH, dW, padH, padW, dilationH, dilationW, group,
                    deformable_group):
    """Host-side restatement of the argument checks the reference runs before a v1 launch (deform_conv_cuda.cpp:62-149);
    returns (batched input, batched offset, batched grad_output, Ho, Wo)."""
    if weight.dim() != 4:
        raise RuntimeError(f"4D weight tensor (nOutputPlane,nInputPlane,kH,kW) expected, but got: {weight.dim()}")
    if not weight.is_contiguous():
        raise RuntimeError("weight tensor has to be contiguous")
    if kW <= 0 or kH <= 0:
        raise RuntimeError(f"kernel size should be greater than zero, but got kH: {kH} kW: {kW}")
    if (weight.size(2), weight.size(3)) != (kH, kW):
        raise RuntimeError(f"kernel size should be consistent with weight, but got kH: {kH} kW: {kW} "
                           f"weight.size(2): {weight.size(2)}, weight.size(3): {weight.size(3)}")
    if dW <= 0 or dH <= 0:
        raise RuntimeError(f"stride should be greater than zero, but got dH: {dH} dW: {dW}")
    if dilationW <= 0 or dilationH <= 0:
        raise RuntimeError(f"dilation should be greater than 0, but got dilationH: {dilationH} dilationW: {dilationW}")
    if input.dim() not in (3, 4):
        raise RuntimeError(f"3D or 4D input tensor expected but got: {input.dim()}")
    if input.dim() == 3:                                    # unbatched call: deform_conv_cuda.cpp:176-183
        input, offset = input.unsqueeze(0), offset.unsqueeze(0)
        if grad_output is not None:
            grad_output = grad_output.unsqueeze(0)
    n_in, n_out = weight.size(1) * group, weight.size(0)
    H, W = input.size(2), input.size(3)
    Ho = (H + 2 * padH - (dilationH * (kH - 1) + 1)) // dH + 1
    Wo = (W + 2 * padW - (dilationW * (kW - 1) + 1)) // dW + 1
    if n_in % deformable_group:
        raise RuntimeError("input channels must divide deformable group size")
    if Wo < 1 or Ho < 1:
        raise RuntimeError(f"Given input size: ({n_in} x {H} x {W}). Calculated output size: ({n_out} x {Ho} x {Wo}). "
                           "Output size is too small")
    if input.size(1) != n_in:
        raise RuntimeError(f"invalid number of input planes, expected: {n_in}, but got: {input.size(1)}")
    if H < kH or W < kW:
        raise RuntimeError("input image is smaller than kernel")
    if (offset.size(2), offset.size(3)) != (Ho, Wo):
        raise RuntimeError(f"invalid spatial size of offset, expected height: {Ho} width: {Wo}, but got height: "
                           f"{offset.size(2)} width: {offset.size(3)}")
    if offset.size(1) != deformable_group * 2 * kH * kW:
        raise RuntimeError("invalid number of channels of offset")
    if offset.size(0) != input.size(0):
        raise RuntimeError("invalid batch size of offset")                       # deform_conv_cuda.cpp:190
    if grad_output is not None:
        if grad_output.size(1) != n_out:
            raise RuntimeError(f"invalid number of gradOutput planes, expected: {n_out}, but got: {grad_output.size(1)}")
        if (grad_output.size(2), grad_output.size(3)) != (Ho, Wo):
            raise RuntimeError(f"invalid size of gradOutput, expected height: {Ho} width: {Wo} , but got height: "
                               f"{grad_output.size(2)} width: {grad_output.size(3)}")
    return input, offset, grad_output, Ho, Wo


def _out_buf(t, accumulate=False):
    """fp32 contiguous view of a caller-owned output (itself when it already is one) and whether to copy back."""
    if t.dtype == torch.float32 and t.is_contiguous():
        return t, False
    return (t.float().contiguous() if accumulate else torch.empty(t.shape, dtype=torch.float32, device=t.device)), True


def deform_conv_forward(input, weight, offset, output, columns, ones, kW, kH, dW, dH, padW, padH, dilationW, dilationH,
                        group, deformable_group, im2col_step):
    """deform_conv_ext.cpp:51-67 -> deform_conv_forward_cuda (deform_conv_cuda.cpp:152-237).  `columns` / `ones` are the
    reference's scratch handles (ignored); `im2col_step` only has to divide the batch (no effect on the result).
    Resizes `output` to [N, Cout, Ho, Wo] like the reference's view/resize dance and returns 1."""
    _check_cuda(input, "deform conv")
    input4, offset4, _, Ho, Wo = _v1_shape_check(input, offset, None, weight, kH, kW, dH, dW, padH, padW, dilationH,
                                                 dilationW, group, deformable_group)
    N, C, H, W = input4.shape
    if N % im2col_step:
        raise RuntimeError("im2col step must divide batchsize")                  # deform_conv_cuda.cpp:189
    Cout = weight.shape[0]
    f64 = _all_f64(input4, weight, offset4, output)
    x, w, off = (input4.contiguous(), weight, offset4.contiguous()) if f64 else (_f32(input4), _f32(weight), _f32(offset4))
    shape = (N, Cout, Ho, Wo) if input.dim() == 4 else (Cout, Ho, Wo)
    if tuple(output.shape) != shape:
        output.resize_(shape)
    if group > 1:           # deform_conv_cuda.cpp:213-226: one GEMM per weight group; composed from per-group calls
        from .ops import group_slices
        parts = []
        for gi in range(group):
            cs, os_, fs, _ms, dgg = group_slices(C, Cout, kH * kW, group, deformable_group, gi)
            part = torch.empty(N, Cout // group, Ho, Wo, dtype=x.dtype, device=input.device)
            deform_conv_forward(x[:, cs].contiguous(), w[os_].contiguous(), off[:, fs].contiguous(), part, columns, ones, kW, kH,
                                dW, dH, padW, padH, dilationW, dilationH, 1, dgg, im2col_step)
            parts.append(part)
        output.copy_(torch.cat(parts, 1).reshape(shape))
        return 1
    if f64:
        out64 = output if output.is_contiguous() else torch.empty(output.shape, dtype=torch.float64, device=output.device)
        with torch.cuda.device(input.device):
            L.check(L.lib().eb_dcn1_forward_f64(L.ptr(x), L.ptr(off), L.ptr(w), L.ptr(out64), N, C, H, W, Cout, kH, kW, dH,
                                                dW, padH, padW, dilationH, dilationW, group, deformable_group,
                                                L.stream_ptr()), "eb_dcn1_forward_f64")
        if out64 is not output:
            output.copy_(out64)
        return 1
    out32, copy_back = _out_buf(output)
    need = L.lib().eb_mdcn_forward_workspace(N, C, H, W, Cout, kH, kW)
    ws = torch.empty(max(need, 16), dtype=torch.uint8, device=input.device)
    with torch.cuda.device(input.device):
        L.check(L.lib().eb_dcn1_forward(L.ptr(x), L.ptr(off), L.ptr(w), L.ptr(out32), N, C, H, W, Cout, kH, kW, dH, dW,
                                        padH, padW, dilationH, dilationW, group, deformable_group, L.ptr(ws), ws.numel(),
                                        L.stream_ptr()), "eb_dcn1_forward")
    if copy_back:
        output.copy_(out32)
    return 1


def deform_conv_backward_input(input, offset, gradOutput, gradInput, gradOffset, weight, columns, kW, kH, dW, dH, padW,
                               padH, dilationW, dilationH, group, deformable_group, im2col_step):
    """deform_conv_ext.cpp:69-86 -> deform_conv_backward_input_cuda (deform_conv_cuda.cpp:239-351): OVERWRITES the caller's
    gradInput and gradOffset; returns 1."""
    _check_cuda(input, "deform conv")
    input4, offset4, go4, Ho, Wo = _v1_shape_check(input, offset, gradOutput, weight, kH, kW, dH, dW, padH, padW,
                                                   dilationH, dilationW, group, deformable_group)
    N, C, H, W = input4.shape
    if N % im2col_step:
        raise RuntimeError("im2col step must divide batchsize")
    Cout = weight.shape[0]
    f64 = _all_f64(input4, offset4, go4, gradInput, gradOffset, weight)
    x, w, off = (input4.contiguous(), weight, offset4.contiguous()) if f64 else (_f32(input4), _f32(weight), _f32(offset4))
    if group > 1:           # composed from per-group calls; deformable groups shared between weight groups accumulate
        from .ops import group_slices
        gx4 = torch.empty(input4.shape, dtype=x.dtype, device=input.device)
        goff4 = torch.zeros(offset4.shape, dtype=x.dtype, device=input.device)
        go4f = go4.to(x.dtype)
        for gi in range(group):
            cs, os_, fs, _ms, dgg = group_slices(C, Cout, kH * kW, group, deformable_group, gi)
            xg, og = x[:, cs].contiguous(), off[:, fs].contiguous()
            gxg, gog = torch.empty_like(xg), torch.empty_like(og)
            deform_conv_backward_input(xg, og, go4f[:, os_].contiguous(), gxg, gog, w[os_].contiguous(), columns, kW, kH, dW, dH,
                                       padW, padH, dilationW, dilationH, 1, dgg, im2col_step)
            gx4[:, cs] = gxg
            goff4[:, fs] += gog
        gradInput.copy_(gx4.reshape(gradInput.shape))
        gradOffset.copy_(goff4.reshape(gradOffset.shape))
        return 1
    if f64:
        gx, goff = torch.empty(input4.shape, dtype=torch.float64, device=input.device), torch.empty_like(off)
        need = L.lib().eb_dcn1_backward_input_f64_workspace(N, C, H, W, Cout, kH, kW, dH, dW, padH, padW, dilationH, dilationW)
        ws = torch.empty(max(need, 16), dtype=torch.uint8, device=input.device)
        with torch.cuda.device(input.device):
            L.check(L.lib().eb_dcn1_backward_input_f64(L.ptr(x), L.ptr(off), L.ptr(w), L.ptr(go4.contiguous()), L.ptr(gx),
                                                       L.ptr(goff), N, C, H, W, Cout, kH, kW, dH, dW, padH, padW, dilationH,
                                                       dilationW, group, deformable_group, L.ptr(ws), ws.numel(),
                                                       L.stream_ptr()), "eb_dcn1_backward_input_f64")
        gradInput.copy_(gx.reshape(gradInput.shape))
        gradOffset.copy_(goff.reshape(gradOffset.shape))
        return 1
    sc = _pow2_scale(go4)
    go = (go4.float() * sc).contiguous()
    gx = torch.empty(gradInput.shape, dtype=torch.float32, device=gradInput.device)
    goff = torch.empty(gradOffset.shape, dtype=torch.float32, device=gradOffset.device)
    need = L.lib().eb_dcn1_backward_workspace(N, C, H, W, Cout, kH, kW, dH, dW, padH, padW, dilationH, dilationW)
    ws = torch.empty(max(need, 16), dtype=torch.uint8, device=input.device)
    with torch.cuda.device(input.device):
        L.check(L.lib().eb_dcn1_backward_input(L.ptr(x), L.ptr(off), L.ptr(w), L.ptr(go), L.ptr(gx), L.ptr(goff), N, C, H, W,
                                               Cout, kH, kW, dH, dW, padH, padW, dilationH, dilationW, group,
                                               deformable_group, L.ptr(ws), ws.numel(), L.stream_ptr()),
                "eb_dcn1_backward_input")
    gradInput.copy_(gx / sc)
    gradOffset.copy_(goff / sc)
    return 1


def deform_conv_backward_parameters(input, offset, gradOutput, gradWeight, columns, ones, kW, kH, dW, dH, padW, padH,
                                    dilationW, dilationH, group, deformable_group, scale, im2col_step):
    """deform_conv_ext.cpp:88-104 -> deform_conv_backward_parameters_cuda (deform_conv_cuda.cpp:353-488):
    gradWeight += scale * dL/dW (accumulated into the caller's tensor); returns 1."""
    _check_cuda(input, "deform conv")
    input4, offset4, go4, Ho, Wo = _v1_shape_check(input, offset, gradOutput, gradWeight, kH, kW, dH, dW, padH, padW,
                                                   dilationH, dilationW, group, deformable_group)
    N, C, H, W = input4.shape
    if N % im2col_step:
        raise RuntimeError("im2col step must divide batchsize")
    Cout = gradWeight.shape[0]
    f64 = _all_f64(input4, offset4, go4, gradWeight)
    x, off = (input4.contiguous(), offset4.contiguous()) if f64 else (_f32(input4), _f32(offset4))
    if group > 1:           # deform_conv_cuda.cpp:455-470 per weight group; composed from per-group calls
        from .ops import group_slices
        go4f = go4.to(x.dtype)
        for gi in range(group):
            cs, os_, fs, _ms, dgg = group_slices(C, Cout, kH * kW, group, deformable_group, gi)
            gwg = torch.zeros(gradWeight[os_].shape, dtype=x.dtype, device=gradWeight.device)
            deform_conv_backward_parameters(x[:, cs].contiguous(), off[:, fs].contiguous(), go4f[:, os_].contiguous(), gwg,
                                            columns, ones, kW, kH, dW, dH, padW, padH, dilationW, dilationH, 1, dgg, scale,
                                            im2col_step)
            gradWeight[os_] += gwg.to(gradWeight.dtype)
        return 1
    if f64:
        gw = torch.zeros(gradWeight.shape, dtype=torch.float64, device=gradWeight.device)
        need = L.lib().eb_dcn1_backward_parameters_f64_workspace(N, C, H, W, Cout, kH, kW, dH, dW, padH, padW, dilationH,
                                                                 dilationW)
        ws = torch.empty(max(need, 16), dtype=torch.uint8, device=input.device)
        with torch.cuda.device(input.device):
            L.check(L.lib().eb_dcn1_backward_parameters_f64(L.ptr(x), L.ptr(off), L.ptr(go4.contiguous()), L.ptr(gw),
                                                            float(scale), N, C, H, W, Cout, kH, kW, dH, dW, padH, padW,
                                                            dilationH, dilationW, group, deformable_group, L.ptr(ws),
                                                            ws.numel(), L.stream_ptr()), "eb_dcn1_backward_parameters_f64")
        gradWeight.add_(gw)
        return 1
    sc = _pow2_scale(go4)
    go = (go4.float() * sc).contiguous()
    gw = torch.zeros(gradWeight.shape, dtype=torch.float32, device=gradWeight.device)
    need = L.lib().eb_dcn1_backward_workspace(N, C, H, W, Cout, kH, kW, dH, dW, padH, padW, dilationH, dilationW)
    ws = torch.empty(max(need, 16), dtype=torch.uint8, device=input.device)
    with torch.cuda.device(input.device):
        L.check(L.lib().eb_dcn1_backward_parameters(L.ptr(x), L.ptr(off), L.ptr(go), L.ptr(gw), float(scale), N, C, H, W,
                                                    Cout, kH, kW, dH, dW, padH, padW, dilationH, dilationW, group,
                                                    deformable_group, L.ptr(ws), ws.numel(), L.stream_ptr()),
                "eb_dcn1_backward_parameters")
    gradWeight.add_((gw / sc).to(gradWeight.dtype))
    return 1
