"""Thin Python front-end over the C ABI: NHWC fp16 views, weight packing, one function per kernel.

PyTorch is used only for device memory and the current CUDA stream; every compute call goes
through libedvr_b200.so (edvr_b200/_lib.py) with raw pointers.
"""
import ctypes
import os

import torch

from . import _lib as L
from ._lib import ACT_LRELU, ACT_NONE, ACT_RELU, ACT_SIGMOID, OUT_PIXSHUF2, OUT_SAME, OUT_STRIDE2  # noqa: F401


LAUNCHES = [0]      # number of libedvr_b200 kernel launches issued through this module (bench.py: gpu_launches)
USE_PAIR = True     # route eligible convolutions to the CTA-pair kernel (conv_pair.cuh)
PROFILE = None      # when a list: (kernel name, algorithmic FLOPs, start event, end event, detail) per call (bench.py)


class _Rec:
    """Counts launches and, when PROFILE is a list, brackets the call with CUDA events on the current stream."""

    def __init__(self, name, kernels=1, flops=0.0, detail=""):
        self.name, self.kernels, self.flops, self.detail = name, kernels, flops, detail

    def __enter__(self):
        LAUNCHES[0] += self.kernels
        if PROFILE is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if PROFILE is not None:
            self.e1.record()
            PROFILE.append((self.name, self.flops, self.e0, self.e1, self.detail))
        return False


class View:
    """Channel slice [ch_off, ch_off+C) of an NHWC fp16 tensor t[N, H, W, Ctot]."""

    __slots__ = ("t", "ch_off", "C")

    def __init__(self, t, ch_off=0, C=None):
        assert t.dtype in (torch.float16, torch.bfloat16) and t.dim() == 4 and t.is_contiguous() and t.is_cuda
        self.t, self.ch_off = t, ch_off
        self.C = t.shape[3] - ch_off if C is None else C
        assert 0 <= ch_off and ch_off + self.C <= t.shape[3]

    N = property(lambda s: s.t.shape[0])
    H = property(lambda s: s.t.shape[1])
    W = property(lambda s: s.t.shape[2])
    pix_stride = property(lambda s: s.t.shape[3])

    def slice(self, off, C):
        return View(self.t, self.ch_off + off, C)

    def dense(self):
        """Materialise as a dense torch tensor [N,H,W,C] (tests / debugging)."""
        return self.t[..., self.ch_off:self.ch_off + self.C]


def new_act(N, H, W, C, device="cuda"):
    return View(torch.empty(N, H, W, C, dtype=torch.float16, device=device))


class PackedConv:
    """MMA-ready fp16 weights + fp32 bias of one convolution (see eb_pack_weight)."""

    __slots__ = ("w", "b", "BN", "n_tiles", "cin", "ksize", "cout", "wpair", "cin_real")


def _choose_bn(cout_packed):
    if cout_packed % 128 == 0:
        return 128
    for bn in (96, 64, 32):
        if cout_packed % bn == 0:
            return bn
    raise ValueError(f"packed Cout {cout_packed} must be a multiple of 32")


def pack_conv(weight, bias=None, cout_packed=None):
    """weight: fp32 [Cout, Cin, k, k] (CUDA)."""
    assert weight.is_cuda and weight.dtype == torch.float32
    weight = weight.contiguous()
    cout, cin, k, _ = weight.shape
    cout_packed = cout_packed or ((cout + 31) // 32) * 32
    p = PackedConv()
    p.BN = _choose_bn(cout_packed)
    p.n_tiles = cout_packed // p.BN
    p.cin, p.ksize, p.cout = cin, k, cout
    p.cin_real = cin        # input channels that carry data (conv_first runs on a zero-padded 64-channel input): FLOP accounting
    nbytes = L.lib().eb_packed_weight_bytes(cin, k * k, p.BN, p.n_tiles)
    p.w = torch.empty(nbytes // 2, dtype=torch.float16, device=weight.device)
    with _Rec("pack_weight", 1):
        L.check(L.lib().eb_pack_weight(L.ptr(weight), cout, cin, k * k, p.BN, p.n_tiles, L.ptr(p.w), L.stream_ptr()),
                "eb_pack_weight")
    p.wpair = None
    if L.lib().eb_conv2d_pair_supported(cin, k, p.BN, p.n_tiles):
        # second packing for the CTA-pair kernel (weights resident in shared memory), see conv_pair.cuh
        p.wpair = torch.empty(nbytes // 2, dtype=torch.float16, device=weight.device)
        with _Rec("pack_weight", 1):
            L.check(L.lib().eb_pack_weight_pair(L.ptr(weight), cout, cin, k * k, p.BN, p.n_tiles,
                                                L.ptr(p.wpair), L.stream_ptr()), "eb_pack_weight_pair")
    b = torch.zeros(cout_packed, dtype=torch.float32, device=weight.device)
    if bias is not None:
        b[:cout] = bias.float()
    p.b = b
    return p


def _src(v, div=1, mul=1, keep=0, add=0):
    return L.Src(v.t.data_ptr(), v.C, v.pix_stride, v.ch_off, div, mul, keep, add)


class Blocked32:
    """fp32 [N,H,W,C] tensor in the library's private tile-blocked layout (eb_f32_blocked_elems)."""

    def __init__(self, N, H, W, C, device="cuda"):
        self.N, self.H, self.W, self.C = N, H, W, C
        n = L.lib().eb_f32_blocked_elems(N, H, W, C)
        self.t = torch.zeros(n, dtype=torch.float32, device=device)

    def to_nhwc(self):
        """Un-block into a dense [N,H,W,C] tensor (tests / debugging only)."""
        N, H, W, C = self.N, self.H, self.W, self.C
        ty, tx = (H + 15) // 16, (W + 15) // 16
        # [tile n, ty, tx][sub 2][q 4][chunk C/32][f4 8][lane 32][e 4]
        v = self.t.view(N, ty, tx, 2, 4, C // 32, 8, 32, 4)
        # lane = (row_in_q 4, col 8); pixel y = q*4 + row_in_q, x = sub*8 + col; channel = chunk*32 + f4*4 + e
        v = v.view(N, ty, tx, 2, 4, C // 32, 8, 4, 8, 4).permute(0, 1, 4, 7, 2, 3, 8, 5, 6, 9)
        v = v.reshape(N, ty * 16, tx * 16, C)
        return v[:, :H, :W, :].contiguous()


def _epi(pc_bias, act, out16=None, out32=None, res16=None, res32=None, out_nchw=None, nchw_C=0,
         out_mode=OUT_SAME, bf16=False):
    e = L.Epilogue()
    e.bf16 = 1 if bf16 else 0
    e.bias = None if pc_bias is None else pc_bias.data_ptr()
    e.act = act
    if res16 is not None:
        e.res16, e.res_pix_stride, e.res_ch_off = res16.t.data_ptr(), res16.pix_stride, res16.ch_off
    if isinstance(res32, Blocked32) or isinstance(out32, Blocked32):
        e.f32_blocked = 1
        if res32 is not None:
            e.res32, e.res_pix_stride, e.res_ch_off = res32.t.data_ptr(), res32.C, 0
        if out32 is not None:
            e.out32, e.out32_pix_stride, e.out32_ch_off = out32.t.data_ptr(), out32.C, 0
        res32 = out32 = None
    if res32 is not None:
        e.res32, e.res_pix_stride, e.res_ch_off = res32.data_ptr(), res32.shape[3], 0
    if out16 is not None:
        e.out16, e.out16_pix_stride, e.out16_ch_off = out16.t.data_ptr(), out16.pix_stride, out16.ch_off
    if out32 is not None:
        e.out32, e.out32_pix_stride, e.out32_ch_off = out32.data_ptr(), out32.shape[3], 0
    if out_nchw is not None:
        e.out_nchw, e.nchw_C = out_nchw.data_ptr(), nchw_C
    e.out_mode = out_mode
    return e


def conv2d(pc, srcs, out16=None, act=ACT_NONE, res16=None, res32=None, out32=None, out_mode=OUT_SAME,
           src_maps=None, N=None, out_nchw=None, nchw_C=0):
    """srcs: list of 1-2 Views (channel-concatenated input). src_maps: per-source (div, mul, keep, add)."""
    v0 = srcs[0]
    N = v0.N if N is None else N
    arr = (L.Src * len(srcs))()
    for i, v in enumerate(srcs):
        m = (1, 1, 0, 0) if src_maps is None or src_maps[i] is None else src_maps[i]
        arr[i] = _src(v, *m)
    assert sum(v.C for v in srcs) == pc.cin, (sum(v.C for v in srcs), pc.cin)
    bf16 = v0.t.dtype == torch.bfloat16
    e = _epi(pc.b, act, out16, out32, res16, res32, out_nchw=out_nchw, nchw_C=nchw_C, out_mode=out_mode, bf16=bf16)
    opix = N * v0.H * v0.W if out_mode != OUT_STRIDE2 else N * ((v0.H + 1) // 2) * ((v0.W + 1) // 2)
    detail = ""
    if PROFILE is not None:
        detail = (f"{pc.cin}->{pc.cout} {N}x{v0.H}x{v0.W} act{act} mode{out_mode}"
                  f"{' res16' if res16 is not None else ''}{' res32' if res32 is not None else ''}"
                  f"{' out32' if out32 is not None else ''}")
    with _Rec(f"conv_igemm_{pc.ksize}x{pc.ksize}", 1, 2.0 * opix * pc.cout * pc.cin_real * pc.ksize * pc.ksize, detail):
        if pc.wpair is not None and USE_PAIR and os.environ.get("EDVR_B200_CONV_PAIR", "1") != "0":
            L.check(L.lib().eb_conv2d_pair(arr, len(srcs), N, v0.H, v0.W, pc.ksize, L.ptr(pc.wpair), pc.BN, pc.n_tiles,
                                           ctypes.byref(e), L.stream_ptr()), "eb_conv2d_pair")
        else:
            L.check(L.lib().eb_conv2d(arr, len(srcs), N, v0.H, v0.W, pc.ksize, L.ptr(pc.w), pc.BN, pc.n_tiles,
                                      ctypes.byref(e), L.stream_ptr()), "eb_conv2d")


class OffsetMonitor:
    """Deferred form of the reference's per-call check `if mean(|offset|) > 50: logger.warning(...)` (arch_util.py:249-253).
    The reference reads the mean back on every DCN call (a device->host sync, 28 per EDVR-L forward); here the kernels add
    sum |offset| into a device accumulator, submit() queues an asynchronous copy of it, and poll() - called at the start of
    the next forward - emits the same warning text for every finished copy.  Nothing ever blocks the stream."""

    def __init__(self):
        self.pending = []

    def submit(self, acc, counts, names=None):
        """acc: device fp32 [k] of sum |offset|; counts: number of offset values behind each entry."""
        host = torch.empty(acc.shape, dtype=torch.float32, pin_memory=True)
        host.copy_(acc, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self.pending.append((host, [float(c) for c in counts], names, ev))
        if len(self.pending) > 64:
            self.poll(block=True)

    def poll(self, block=False):
        """Warn for every completed check; returns the list of means seen (oldest first)."""
        import logging
        seen = []
        while self.pending and (block or self.pending[0][3].query()):
            host, counts, names, ev = self.pending.pop(0)
            ev.synchronize()
            for i, c in enumerate(counts):
                mean = float(host[i]) / max(c, 1.0)
                seen.append(mean)
                if mean > 50:
                    logging.getLogger("basicsr").warning(f"Offset abs mean is {mean}, larger than 50.")
        return seen


class DcnSite:
    """One DCNv2Pack site (arch_util.py:232-257): conv_offset -> (offset, sigmoid(mask)) -> modulated deformable conv.

    wo/bo: conv_offset weight [dg*27, C, 3, 3] / bias, w/b: DCN weight [Cout, C, 3, 3] / bias (reference state_dict tensors).
    __call__(x, feat, out16, act, absmean): x = features to sample, feat = offset features, both NHWC fp16 Views.

    mode "pair" (default): ONE launch of the CTA-pair kernel (dcn_pair.cuh): conv_offset runs on the tensor cores inside the
    DCN kernel, overlapped with the gather; offsets and masks stay in tensor memory.  mode "fused": the single-CTA form of
    the same fusion (dcn_site.cuh; odd dg, more than one output-channel tile).  mode "split": conv_offset as a separate convolution writing the reference's fp32 NCHW
    offset/mask-logit tensor, then the same DCN kernel reading it (used when dg*27 > 224).  `mode` (default: the
    EDVR_B200_DCN_SITE environment variable, else "pair") is where the selection starts; a site that the requested kernel
    cannot serve moves on to the next mode of pair -> fused -> split."""

    MODES = ("pair", "fused", "split")

    def __init__(self, wo, bo, w, b, dg, mode=None):
        mode = mode or os.environ.get("EDVR_B200_DCN_SITE", "pair")
        if mode not in self.MODES:
            raise ValueError(f"DcnSite mode {mode!r}: expected one of {', '.join(self.MODES)}")
        self.dg = dg
        self.C = w.shape[1]
        self.main = pack_conv(w, b)
        if mode == "pair" and not (w.shape[2] == 3 and self.main.wpair is not None and
                                   L.lib().eb_dcn_pair_supported(self.C, dg, self.main.BN, self.main.n_tiles)):
            mode = "fused"
        if mode == "fused" and (dg * 27 > 224 or w.shape[2] != 3):
            mode = "split"
        self.mode = mode
        self.n_off = dg * 27
        if mode == "pair":
            nbytes = L.lib().eb_dcn_pair_offset_weight_bytes(self.C)
            self.wo_pack = torch.empty(nbytes // 2, dtype=torch.float16, device=w.device)
            self.bo_cols = torch.empty(224, dtype=torch.float32, device=w.device)
            with _Rec("pack_weight", 1):
                L.check(L.lib().eb_dcn_pair_pack_offset_weight(L.ptr(wo.contiguous()), L.ptr(None if bo is None else bo.contiguous()),
                                                               self.C, dg, L.ptr(self.wo_pack), L.ptr(self.bo_cols),
                                                               L.stream_ptr()), "eb_dcn_pair_pack_offset_weight")
        elif mode == "fused":
            nbytes = L.lib().eb_dcn_site_offset_weight_bytes(self.C)
            self.wo_pack = torch.empty(nbytes // 2, dtype=torch.float16, device=w.device)
            self.bo_cols = torch.empty(224, dtype=torch.float32, device=w.device)
            with _Rec("pack_weight", 1):
                L.check(L.lib().eb_dcn_site_pack_offset_weight(L.ptr(wo.contiguous()), L.ptr(None if bo is None else bo.contiguous()),
                                                               self.C, dg, L.ptr(self.wo_pack), L.ptr(self.bo_cols),
                                                               L.stream_ptr()), "eb_dcn_site_pack_offset_weight")
        else:
            self.offset = pack_conv(wo, bo, cout_packed=((dg * 27 + 127) // 128) * 128)
        self._rec = {}

    def _raw(self, N, H, W, device):
        key = (N, H, W)
        t = self._rec.get(key)
        if t is None:
            self._rec.clear()           # one shape at a time: the offsets are the largest temporary of the graph
            t = torch.empty(N, self.n_off, H, W, dtype=torch.float32, device=device)
            self._rec[key] = t
        return t

    def arena_record(self, arena, feat):
        """Scratch for the offsets shared by all sites of an executor (engine._Arena); None when nothing is materialised."""
        if self.mode != "split":
            return None
        return arena.f32("offraw", feat.N, self.n_off, feat.H, feat.W)

    def __call__(self, x, feat, out16=None, act=ACT_NONE, absmean=None, record=None, out_nchw=None):
        """out16: NHWC fp16 View, or out_nchw: fp32 [N, Cout, H, W] (the reference operator's layout)."""
        N, H, W = feat.N, feat.H, feat.W
        pc = self.main
        flops = 2.0 * N * H * W * pc.cout * pc.cin * 9
        e = _epi(pc.b, act, out16, out_nchw=out_nchw, nchw_C=pc.cout)
        am = None if absmean is None else absmean.data_ptr()
        if self.mode == "pair":
            with _Rec("dcn_site", 1, flops + 2.0 * N * H * W * self.n_off * pc.cin * 9, f"{N}x{H}x{W} C{x.C} pair"):
                L.check(L.lib().eb_dcn_site_pair(L.ptr(x.t), x.pix_stride, x.ch_off, N, H, W, x.C, self.dg,
                                                 L.ptr(feat.t), feat.pix_stride, feat.ch_off, L.ptr(self.wo_pack),
                                                 L.ptr(self.bo_cols), L.ptr(pc.wpair), pc.BN, ctypes.byref(e), am,
                                                 L.stream_ptr()), "eb_dcn_site_pair")
            return
        if self.mode == "split":
            raw = record if record is not None else self._raw(N, H, W, feat.t.device)
            conv2d(self.offset, [feat], act=ACT_NONE, out_nchw=raw, nchw_C=self.n_off)
            plane = H * W
            off_ptr = raw.data_ptr()
            with _Rec("dcn_site", 1, flops, f"{N}x{H}x{W} C{x.C} split"):
                L.check(L.lib().eb_dcn_site(L.ptr(x.t), x.pix_stride, x.ch_off, N, H, W, x.C, self.dg,
                                            off_ptr, off_ptr + self.dg * 18 * plane * 4, self.n_off * plane, self.n_off * plane, 1,
                                            None, 0, 0, None, None, L.ptr(pc.w), pc.BN, pc.n_tiles, ctypes.byref(e), am,
                                            L.stream_ptr()), "eb_dcn_site")
            return
        with _Rec("dcn_site", 1, flops + 2.0 * N * H * W * self.n_off * pc.cin * 9, f"{N}x{H}x{W} C{x.C} fused"):
            L.check(L.lib().eb_dcn_site(L.ptr(x.t), x.pix_stride, x.ch_off, N, H, W, x.C, self.dg,
                                        None, None, 0, 0, 1, L.ptr(feat.t), feat.pix_stride, feat.ch_off,
                                        L.ptr(self.wo_pack), L.ptr(self.bo_cols), L.ptr(pc.w), pc.BN, pc.n_tiles,
                                        ctypes.byref(e), am, L.stream_ptr()), "eb_dcn_site")


def nchw_to_nhwc(x, out=None):
    """fp32 [N,C,H,W] -> View fp16 [N,H,W,C]."""
    N, C, H, W = x.shape
    out = out or new_act(N, H, W, C, x.device)
    with _Rec("layout", 1):
        L.check(L.lib().eb_nchw_f32_to_nhwc_f16(L.ptr(x.contiguous()), L.ptr(out.t), N, C, H, W, out.pix_stride,
                                                out.ch_off, L.stream_ptr()), "eb_nchw_f32_to_nhwc_f16")
    return out


def nhwc_to_nchw(v):
    out = torch.empty(v.N, v.C, v.H, v.W, dtype=torch.float32, device=v.t.device)
    with _Rec("layout", 1):
        L.check(L.lib().eb_nhwc_f16_to_nchw_f32(L.ptr(v.t), v.pix_stride, v.ch_off, L.ptr(out), v.N, v.C, v.H, v.W,
                                                L.stream_ptr()), "eb_nhwc_f16_to_nchw_f32")
    return out


def conv_first(x_nchw, w, b, out, act=ACT_LRELU):
    N, _, H, W = x_nchw.shape
    with _Rec("conv_first", 1):
        L.check(L.lib().eb_conv_first(L.ptr(x_nchw), L.ptr(w), L.ptr(b), L.ptr(out.t), N, H, W, w.shape[0],
                                      out.pix_stride, act, L.stream_ptr()), "eb_conv_first")


def add_base(base, base_img_stride, scale, out_nchw):
    """out_nchw (fp32 [N,C,H,W]) += bilinear x4 of base (scale 4) or base (scale 1)."""
    N, C, H, W = out_nchw.shape
    with _Rec("add_base", 1):
        L.check(L.lib().eb_add_base(L.ptr(base), base_img_stride, scale, L.ptr(out_nchw), N, C, H, W, L.stream_ptr()),
                "eb_add_base")


def conv_last(x, w, b, base, base_img_stride, scale, out_nchw):
    with _Rec("conv_last", 1):
        L.check(L.lib().eb_conv_last(L.ptr(x.t), x.pix_stride, L.ptr(w), L.ptr(b), L.ptr(base), base_img_stride, scale,
                                     L.ptr(out_nchw), x.N, x.H, x.W, x.C, L.stream_ptr()), "eb_conv_last")


def upsample2x(src, dst, mul=1.0, add=None):
    a = (None, 0, 0) if add is None else (add.t, add.pix_stride, add.ch_off)
    with _Rec("upsample2x", 1):
        L.check(L.lib().eb_upsample2x(L.ptr(src.t), src.pix_stride, src.ch_off, L.ptr(dst.t), dst.pix_stride, dst.ch_off,
                                      src.N, src.H, src.W, src.C, mul, L.ptr(a[0]), a[1], a[2], L.stream_ptr()),
                "eb_upsample2x")


def pool_max_avg(src, dst):
    with _Rec("pool", 1):
        L.check(L.lib().eb_pool_max_avg(L.ptr(src.t), src.pix_stride, src.ch_off, L.ptr(dst.t), dst.pix_stride,
                                        dst.ch_off, src.N, src.H, src.W, src.C, L.stream_ptr()), "eb_pool_max_avg")


def tsa_temporal(emb, emb_ref, aligned, dst, B, T):
    with _Rec("tsa_temporal", 1):
        L.check(L.lib().eb_tsa_temporal(L.ptr(emb.t), L.ptr(emb_ref.t), L.ptr(aligned.t), L.ptr(dst.t), B, T, emb.H,
                                        emb.W, emb.C, L.stream_ptr()), "eb_tsa_temporal")


def tsa_modulate(feat, attn, attn_add, out16=None, out32=None):
    blocked = isinstance(out32, Blocked32)
    o32 = out32.t if blocked else out32
    with _Rec("tsa_modulate", 1):
        L.check(L.lib().eb_tsa_modulate(L.ptr(feat.t), feat.pix_stride, feat.ch_off, L.ptr(attn.t), L.ptr(attn_add.t),
                                        L.ptr(None if out16 is None else out16.t), L.ptr(o32), attn.N, attn.H, attn.W,
                                        attn.C, 1 if blocked else 0, L.stream_ptr()), "eb_tsa_modulate")


def group_slices(C, Cout, K, groups, dg, gi):
    """Weight group gi of a grouped (deformable) convolution as a groups == 1 problem: (input channels, output channels,
    offset channels, mask channels, deformable groups of the slice).  The reference runs one im2col over all channels and
    one GEMM per weight group (deform_conv_cuda.cpp:536-568); its column rows of group gi belong to the deformable groups
    below, which are whole groups when dg % groups == 0 and one shared group when groups % dg == 0."""
    Cg, Og = C // groups, Cout // groups
    if dg % groups == 0:
        dgg = dg // groups
        d0 = gi * dgg
    elif groups % dg == 0:
        dgg, d0 = 1, gi // (groups // dg)
    else:
        raise RuntimeError(f"edvr_b200: groups={groups} with deformable_groups={dg} (one must divide the other)")
    return (slice(gi * Cg, (gi + 1) * Cg), slice(gi * Og, (gi + 1) * Og), slice(d0 * 2 * K, (d0 + dgg) * 2 * K),
            slice(d0 * K, (d0 + dgg) * K), dgg)


def mdcn_forward(x, offset, mask, weight, bias, stride, padding, dilation, groups, dg, workspace=None):
    """Reference-layout operator (fp32 NCHW) through eb_mdcn_forward, or through eb_mdcn_forward_f64 when x is float64
    (then every tensor is float64 and contiguous).  Weight groups > 1 (deform_conv_cuda.cpp:536-568) are composed from
    per-group calls on channel slices - EDVR itself always uses groups == 1."""
    N, C, H, W = x.shape
    Cout, _, kh, kw = weight.shape
    if groups > 1:
        outs = []
        for gi in range(groups):
            cs, os_, fs, ms, dgg = group_slices(C, Cout, kh * kw, groups, dg, gi)
            outs.append(mdcn_forward(x[:, cs].contiguous(), offset[:, fs].contiguous(), mask[:, ms].contiguous(),
                                     weight[os_].contiguous(), None if bias is None else bias[os_].contiguous(),
                                     stride, padding, dilation, 1, dgg))
        return torch.cat(outs, 1)
    Ho = (H + 2 * padding - (dilation * (kh - 1) + 1)) // stride + 1
    Wo = (W + 2 * padding - (dilation * (kw - 1) + 1)) // stride + 1
    if x.dtype == torch.float64:
        out = torch.empty(N, Cout, Ho, Wo, dtype=torch.float64, device=x.device)
        with _Rec("mdcn_forward_f64", 1):
            L.check(L.lib().eb_mdcn_forward_f64(L.ptr(x), L.ptr(offset), L.ptr(mask), L.ptr(weight), L.ptr(bias),
                                                L.ptr(out), N, C, H, W, Cout, kh, kw, stride, padding, dilation, groups,
                                                dg, L.stream_ptr()), "eb_mdcn_forward_f64")
        return out
    out = torch.empty(N, Cout, Ho, Wo, dtype=torch.float32, device=x.device)
    need = L.lib().eb_mdcn_forward_workspace(N, C, H, W, Cout, kh, kw)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(max(need, 16), dtype=torch.uint8, device=x.device)
    with _Rec("mdcn_forward_op", 4):
        L.check(L.lib().eb_mdcn_forward(L.ptr(x), L.ptr(offset), L.ptr(mask), L.ptr(weight), L.ptr(bias), L.ptr(out),
                                        N, C, H, W, Cout, kh, kw, stride, padding, dilation, groups, dg,
                                        L.ptr(workspace), workspace.numel(), L.stream_ptr()), "eb_mdcn_forward")
    return out
