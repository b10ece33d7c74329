"""The double-precision deformable-convolution operator (csrc/dcn_f64.cuh, the eb_*_f64 entry points) and its dispatch:
all-fp64 calls of the B1 shim, the autograd Functions and the Pack modules run it end to end in fp64.

Checkers: torch.autograd.gradcheck (finite differences of our own forward), torchvision.ops.deform_conv2d in float64 on
the CPU, and the fp32 outputs of the unmodified reference extension (tests/golden/dcn*_ref_cuda_*.npz).  Sample
coordinates are kept at least 1e-4 away from integers wherever a result is compared against finite differences or
another implementation: bilinear sampling has kinks there, and torchvision differs from the reference at coordinate -1.
The last test runs on the host without a GPU."""
import glob
import math
import os

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
BAR = 1e-11          # max|got - ref| / max|ref| against an fp64 reference


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from edvr_b200 import build
    build.build()
    return torch.device("cuda")


def _err(got, ref):
    got, ref = torch.as_tensor(got).double().cpu(), torch.as_tensor(ref).double().cpu()
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


def _pair(v):
    return (v, v) if isinstance(v, int) else tuple(v)


def _coords(off, kh, kw, stride, pad, dil):
    """Sample coordinates of every offset channel: [N, dg * 2 * kh * kw, Ho, Wo] (h for even channels, w for odd)."""
    (sh, sw), (ph, pw), (dh, dw) = _pair(stride), _pair(pad), _pair(dil)
    N, ch, Ho, Wo = off.shape
    ki, kj = torch.meshgrid(torch.arange(kh), torch.arange(kw), indexing="ij")
    bh = (torch.arange(Ho).view(1, Ho, 1) * sh - ph + ki.reshape(-1, 1, 1) * dh).expand(-1, Ho, Wo)
    bw = (torch.arange(Wo).view(1, 1, Wo) * sw - pw + kj.reshape(-1, 1, 1) * dw).expand(-1, Ho, Wo)
    base = torch.stack((bh, bw), 1).reshape(2 * kh * kw, Ho, Wo).double()
    return off + base.repeat(ch // (2 * kh * kw), 1, 1)


def _off_integers(off, *geom):
    """Moves every offset whose sample coordinate lies within 1e-3 of an integer by 0.01 px."""
    c = _coords(off, *geom)
    return off + 0.01 * ((c - c.round()).abs() < 1e-3).double()


def _assert_off_integers(off, *geom):
    c = _coords(off, *geom)
    assert float((c - c.round()).abs().min()) >= 1e-4


def _case(N, C, H, W, Cout, kh, kw, stride, pad, dil, dg, seed, sigma=2.0, bias=True, groups=1, modulated=True):
    """Seeded fp64 CPU tensors: x, offset (std `sigma` px, coordinates kept off integers), mask, weight, bias."""
    (sh, sw), (ph, pw), (dh, dw) = _pair(stride), _pair(pad), _pair(dil)
    Ho, Wo = (H + 2 * ph - dh * (kh - 1) - 1) // sh + 1, (W + 2 * pw - dw * (kw - 1) - 1) // sw + 1
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, C, H, W, generator=g, dtype=torch.float64)
    off = _off_integers(torch.randn(N, dg * 2 * kh * kw, Ho, Wo, generator=g, dtype=torch.float64) * sigma,
                        kh, kw, stride, pad, dil)
    _assert_off_integers(off, kh, kw, stride, pad, dil)
    mask = torch.rand(N, dg * kh * kw, Ho, Wo, generator=g, dtype=torch.float64) if modulated else None
    w = torch.randn(Cout, C // groups, kh, kw, generator=g, dtype=torch.float64) / math.sqrt(C * kh * kw)
    b = torch.randn(Cout, generator=g, dtype=torch.float64) if bias else None
    return x, off, mask, w, b


def _fp32_kinks(off, *geom):
    """Offsets of the fp32 goldens whose sample coordinate lies within 1e-6 of an integer but not on it (both channels of
    the tap), and their count.  The reference adds the offset to the integer grid position in fp32, which can put such a
    coordinate on the other side of the integer than the exact fp64 sum; grad_offset jumps there (bilinear sampling has a
    kink).  Coordinates exactly on an integer are exact in fp32 too."""
    c = _coords(off, *geom)
    dist = (c - c.round()).abs()
    near = ((dist < 1e-6) & (dist > 0)).reshape(off.shape[0], -1, 2, *off.shape[2:]).any(2, keepdim=True)
    return near.expand(-1, -1, 2, -1, -1).reshape(off.shape), int(near.sum())


# taps with such a coordinate in each golden (found by _fp32_kinks on the recorded offsets); every other golden has none
GOLDEN_KINKS = {"dcn1_ref_cuda_v1_c64_dg8.npz": 1}


def _cuda_leaves(*ts):
    return [None if t is None else t.cuda().requires_grad_() for t in ts]


# ---- 1. gradcheck -----------------------------------------------------------------------------------------------------
# (N, C, H, W, Cout, kh, kw, stride, pad, dil, dg, bias, groups)
V2_GRADCHECK = [
    ("3x3_pad1_dg1_bias", (1, 4, 5, 6, 3, 3, 3, 1, 1, 1, 1, True, 1)),
    ("stride2_dg2_nobias", (2, 4, 5, 6, 3, 3, 3, 2, 1, 1, 2, False, 1)),
    ("dil2_pad2_dg2_bias", (1, 4, 5, 6, 3, 3, 3, 1, 2, 2, 2, True, 1)),
    ("k1x3_dg2_bias", (1, 4, 5, 6, 3, 1, 3, 1, 1, 1, 2, True, 1)),
    ("groups2_dg2_bias", (1, 4, 5, 6, 4, 3, 3, 1, 1, 1, 2, True, 2)),
]
V1_GRADCHECK = [
    ("3x3_pad1_dg1", (1, 4, 5, 6, 3, 3, 3, 1, 1, 1, 1, False, 1)),
    ("aniso_dg2", (1, 4, 5, 6, 3, 3, 3, (1, 2), (1, 0), (2, 1), 2, False, 1)),
    ("k1x3_dg2", (1, 4, 5, 6, 3, 1, 3, 1, (0, 1), 1, 2, False, 1)),
    ("groups2_dg1", (1, 4, 5, 6, 4, 3, 3, 1, 1, 1, 1, False, 2)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,cfg", V2_GRADCHECK, ids=[c[0] for c in V2_GRADCHECK])
def test_gradcheck_modulated_deform_conv(cuda, name, cfg):
    from edvr_b200.dcn import modulated_deform_conv
    N, C, H, W, Cout, kh, kw, s, p, d, dg, bias, groups = cfg
    x, off, mask, w, b = _cuda_leaves(*_case(N, C, H, W, Cout, kh, kw, s, p, d, dg, seed=len(name), bias=bias,
                                             groups=groups))
    fn = lambda x, off, mask, w, *b: modulated_deform_conv(x, off, mask, w, b[0] if b else None, s, p, d, groups, dg)
    # nondet_tol: grad_x is an fp64 atomic scatter, so two backward passes may differ in the last bits
    assert torch.autograd.gradcheck(fn, (x, off, mask, w) + ((b,) if bias else ()), nondet_tol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("name,cfg", V1_GRADCHECK, ids=[c[0] for c in V1_GRADCHECK])
def test_gradcheck_deform_conv(cuda, name, cfg):
    from edvr_b200.dcn import deform_conv
    N, C, H, W, Cout, kh, kw, s, p, d, dg, _bias, groups = cfg
    x, off, _m, w, _b = _case(N, C, H, W, Cout, kh, kw, s, p, d, dg, seed=len(name) + 50, bias=False, groups=groups,
                              modulated=False)
    x, off, w = _cuda_leaves(x, off, w)
    fn = lambda x, off, w: deform_conv(x, off, w, s, p, d, groups, dg)
    # nondet_tol: grad_x is an fp64 atomic scatter, so two backward passes may differ in the last bits
    assert torch.autograd.gradcheck(fn, (x, off, w), nondet_tol=1e-12)


# ---- 2. against torchvision in float64 ------------------------------------------------------------------------------
def _tv(x, off, mask, w, b, stride, pad, dil, go):
    """torchvision forward and gradients on the CPU in float64: out, [grad_x, grad_offset, grad_mask, grad_weight, grad_bias]."""
    from torchvision.ops import deform_conv2d
    leaves = [None if t is None else t.detach().clone().requires_grad_() for t in (x, off, mask, w, b)]
    y = deform_conv2d(leaves[0], leaves[1], leaves[3], leaves[4], stride=_pair(stride), padding=_pair(pad),
                      dilation=_pair(dil), mask=leaves[2])
    y.backward(go)
    return y.detach(), [None if t is None else t.grad for t in leaves]


def _ours(fn_v2, x, off, mask, w, b, go):
    leaves = _cuda_leaves(x, off, mask, w, b)
    y = fn_v2(*leaves)
    y.backward(go.cuda())
    return y.detach(), [None if t is None else t.grad for t in leaves]


TV_CASES = [   # name, (N, C, H, W, Cout, kh, kw, stride, pad, dil, dg), modulated
    ("ragged_v2", (2, 24, 37, 23, 70, 3, 3, 1, 1, 1, 3), True),
    ("edvr_like_v2", (2, 64, 48, 64, 64, 3, 3, 1, 1, 1, 8), True),
    ("ragged_v1_aniso", (2, 24, 37, 23, 70, 3, 3, (2, 1), (1, 2), (1, 2), 3), False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,cfg,modulated", TV_CASES, ids=[c[0] for c in TV_CASES])
def test_forward_and_gradients_vs_torchvision_f64(cuda, name, cfg, modulated):
    from edvr_b200.dcn import deform_conv, modulated_deform_conv
    N, C, H, W, Cout, kh, kw, s, p, d, dg = cfg
    x, off, mask, w, b = _case(N, C, H, W, Cout, kh, kw, s, p, d, dg, seed=7, bias=modulated, modulated=modulated)
    Ho, Wo = off.shape[2:]
    go = torch.randn(N, Cout, Ho, Wo, generator=torch.Generator().manual_seed(8), dtype=torch.float64)
    ref, ref_grads = _tv(x, off, mask, w, b, s, p, d, go)
    if modulated:
        got, grads = _ours(lambda x, o, m, w, b: modulated_deform_conv(x, o, m, w, b, s, p, d, 1, dg), x, off, mask, w, b, go)
    else:
        got, grads = _ours(lambda x, o, m, w, b: deform_conv(x, o, w, s, p, d, 1, dg), x, off, None, w, None, go)
    assert got.dtype == torch.float64 and _err(got, ref) <= BAR, ("out", _err(got, ref))
    for nm, g, r in zip(("grad_x", "grad_offset", "grad_mask", "grad_weight", "grad_bias"), grads, ref_grads):
        if r is None:
            continue
        assert g.dtype == torch.float64 and _err(g, r) <= BAR, (nm, _err(g, r))


# ---- 3. against the reference's semantics ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "dcn_ref_cuda_*.npz"))))
def test_shim_f64_vs_reference_cuda_golden(cuda, path):
    """The fp32 recordings of the unmodified reference extension, fed as fp64 through the B1 shim's v2 pair."""
    from edvr_b200 import deform_conv_ext as ext
    z = np.load(path)
    N, C, H, W, Cout, dg, s, p, d, groups = (int(v) for v in z["meta"])
    t = {k: torch.from_numpy(z[k]).double().cuda() for k in ("x", "offset", "mask", "weight", "bias", "grad_out")}
    kh, kw = t["weight"].shape[2:]
    out = torch.empty(z["out"].shape, dtype=torch.float64, device="cuda")
    e = t["x"].new_empty(0)
    ext.modulated_deform_conv_forward(t["x"], t["weight"], t["bias"], e, t["offset"], t["mask"], out, e, kh, kw, s, s, p, p,
                                      d, d, groups, dg, True)
    assert _err(out, z["out"]) <= 5e-6, ("out", _err(out, z["out"]))
    gx, goff, gm = torch.empty_like(t["x"]), torch.empty_like(t["offset"]), torch.empty_like(t["mask"])
    gw, gb = torch.zeros_like(t["weight"]), torch.zeros_like(t["bias"])
    ext.modulated_deform_conv_backward(t["x"], t["weight"], t["bias"], e, t["offset"], t["mask"], e, gx, gw, gb, goff, gm,
                                       t["grad_out"], kh, kw, s, s, p, p, d, d, groups, dg, True)
    kink, n_kink = _fp32_kinks(t["offset"].cpu(), kh, kw, s, p, d)
    assert n_kink == GOLDEN_KINKS.get(os.path.basename(path), 0)
    goff, ref_goff = goff.cpu()[~kink], torch.from_numpy(z["grad_offset"])[~kink]
    assert _err(goff, ref_goff) <= 5e-6, ("grad_offset", _err(goff, ref_goff))
    for nm, g in (("grad_x", gx), ("grad_mask", gm), ("grad_weight", gw), ("grad_bias", gb)):
        assert g.dtype == torch.float64 and _err(g, z[nm]) <= 5e-6, (nm, _err(g, z[nm]))


@pytest.mark.gpu
@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "dcn1_ref_cuda_*.npz"))))
def test_shim_f64_v1_vs_reference_cuda_golden(cuda, path):
    from edvr_b200 import deform_conv_ext as ext
    z = np.load(path)
    N, C, H, W, Cout, dg, kh, kw, sh, sw, ph, pw, dh, dw = (int(v) for v in z["meta"])
    scale = float(z["scale"])
    x, off, w, go = (torch.from_numpy(z[k]).double().cuda() for k in ("x", "offset", "weight", "grad_out"))
    geom = (kw, kh, sw, sh, pw, ph, dw, dh, 1, dg)
    out, e = x.new_empty(0), x.new_empty(0)
    ext.deform_conv_forward(x, w, off, out, e, e, *geom, N)
    assert out.dtype == torch.float64 and _err(out, z["out"]) <= 5e-6, ("out", _err(out, z["out"]))
    gx, goff = torch.full_like(x, 7.0), torch.full_like(off, 7.0)        # overwritten
    ext.deform_conv_backward_input(x, off, go, gx, goff, w, e, *geom, N)
    gw = torch.ones_like(w)                                              # accumulated into
    ext.deform_conv_backward_parameters(x, off, go, gw, e, e, *geom, scale, N)
    kink, n_kink = _fp32_kinks(off.cpu(), kh, kw, (sh, sw), (ph, pw), (dh, dw))
    assert n_kink == GOLDEN_KINKS.get(os.path.basename(path), 0)
    for nm, g, ref in (("grad_x", gx, z["grad_x"]), ("grad_offset", goff.cpu()[~kink], z["grad_offset"][~kink.numpy()]),
                       ("grad_weight", gw - 1.0, z["grad_weight"])):
        assert _err(g, ref) <= 5e-6, (nm, _err(g, ref))


@pytest.mark.gpu
def test_minus_one_edge_follows_reference(cuda):
    """Zero offsets and padding 1 put every border tap exactly on coordinate -1: grad_offset is exactly 0 there, as in the
    reference (and unlike torchvision), and non-zero inside."""
    from edvr_b200.dcn import _mdcn_backward_raw
    N, C, H, W, Cout, dg = 1, 4, 5, 6, 3, 2
    x, _off, mask, w, _b = _case(N, C, H, W, Cout, 3, 3, 1, 1, 1, dg, seed=1)
    off = torch.zeros(N, dg * 18, H, W, dtype=torch.float64)
    go = torch.randn(N, Cout, H, W, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    _gx, goff, _gm, _gw, _gb = _mdcn_backward_raw(*(t.cuda() for t in (x, off, mask, w, go)), True, 1, 1, 1, 1, dg)
    goff = goff.cpu().reshape(N, dg, 9, 2, H, W)
    assert torch.all(goff[:, :, 0:3, :, 0, :] == 0)             # taps (0, *) at output row 0 sample h = -1
    assert torch.all(goff[:, :, [0, 3, 6], :, :, 0] == 0)       # taps (*, 0) at output column 0 sample w = -1
    assert goff[:, :, 4, :, 2, 2].abs().max() > 0


# ---- 4. determinism ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_repeated_calls_are_bit_identical(cuda):
    """out, grad_offset, grad_mask, grad_weight (split-K over 2 pixel splits, reduced in order) and grad_bias repeat bit
    for bit; grad_x, an atomic scatter, to 1e-14."""
    from edvr_b200 import ops
    from edvr_b200.dcn import _mdcn_backward_raw
    x, off, mask, w, b = (t.cuda() for t in _case(2, 16, 40, 40, 24, 3, 3, 1, 1, 1, 4, seed=11))
    go = torch.randn(2, 24, 40, 40, generator=torch.Generator().manual_seed(12), dtype=torch.float64).cuda()
    runs = []
    for _ in range(2):
        out = ops.mdcn_forward(x, off, mask, w, b, 1, 1, 1, 1, 4)
        runs.append((out,) + _mdcn_backward_raw(x, off, mask, w, go, True, 1, 1, 1, 1, 4))
    (o1, gx1, *rest1), (o2, gx2, *rest2) = runs
    assert torch.equal(o1, o2)
    for nm, a, c in zip(("grad_offset", "grad_mask", "grad_weight", "grad_bias"), rest1, rest2):
        assert torch.equal(a, c), nm
    assert _err(gx1, gx2) <= 1e-14


# ---- 5. dispatch ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_all_f64_calls_run_in_f64_at_every_layer(cuda):
    """The B1 shim, the autograd Function and a .double() DCNv2Pack under no_grad all match torchvision fp64 to 1e-11,
    which the fp16-operand kernels cannot reach."""
    import torch.nn.functional as F
    from edvr_b200 import deform_conv_ext as ext
    from edvr_b200.dcn import DCNv2Pack, modulated_deform_conv
    N, C, H, W, Cout, dg = 1, 64, 12, 14, 64, 8
    x, off, mask, w, b = _case(N, C, H, W, Cout, 3, 3, 1, 1, 1, dg, seed=21)
    ref = _tv(x, off, mask, w, b, 1, 1, 1, torch.zeros(N, Cout, H, W, dtype=torch.float64))[0]
    xc, oc, mc, wc, bc = (t.cuda() for t in (x, off, mask, w, b))
    out = torch.empty(N, Cout, H, W, dtype=torch.float64, device="cuda")
    e = xc.new_empty(0)
    ext.modulated_deform_conv_forward(xc, wc, bc, e, oc, mc, out, e, 3, 3, 1, 1, 1, 1, 1, 1, 1, dg, True)
    assert _err(out, ref) <= BAR, ("shim", _err(out, ref))
    y = modulated_deform_conv(xc, oc, mc, wc, bc, 1, 1, 1, 1, dg)
    assert y.dtype == torch.float64 and _err(y, ref) <= BAR, ("function", _err(y, ref))

    torch.manual_seed(22)
    m = DCNv2Pack(C, Cout, 3, padding=1, deformable_groups=dg).double()
    with torch.no_grad():
        m.conv_offset.weight.normal_(0, 0.05)
        m.conv_offset.bias.normal_(0, 0.5)
        m.bias.normal_(0, 0.1)
    feat = torch.randn(N, C, H, W, generator=torch.Generator().manual_seed(23), dtype=torch.float64)
    o = F.conv2d(feat, m.conv_offset.weight, m.conv_offset.bias, padding=1)
    o1, o2, mk = torch.chunk(o, 3, dim=1)
    ref_pack = _tv(x, torch.cat((o1, o2), 1), torch.sigmoid(mk), m.weight.detach(), m.bias.detach(), 1, 1, 1,
                   torch.zeros(N, Cout, H, W, dtype=torch.float64))[0]
    m = m.cuda()
    with torch.no_grad():
        assert not m._fusable(xc)
        yp = m(xc, feat.cuda())
    assert yp.dtype == torch.float64 and _err(yp, ref_pack) <= BAR, ("DCNv2Pack", _err(yp, ref_pack))


@pytest.mark.gpu
@pytest.mark.parametrize("cls,stride,padding", [("ModulatedDeformConvPack", 1, 0), ("DCNv2Pack", 2, 1)])
def test_fp32_pack_outside_the_fused_geometry_is_not_fused(cuda, cls, stride, padding):
    """The fused DCN site is 3x3 / stride 1 / pad 1 only: an fp32 Pack with padding 0 or stride 2 is not fusable under no_grad
    and returns exactly what its conv_offset followed by the operator returns, at the reference's output size."""
    from edvr_b200 import dcn
    torch.manual_seed(41)
    m = getattr(dcn, cls)(64, 64, 3, stride=stride, padding=padding, deformable_groups=8).cuda()
    with torch.no_grad():
        m.conv_offset.weight.normal_(0, 0.02)
        m.conv_offset.bias.normal_(0, 0.5)
    x = torch.randn(1, 64, 12, 14, device="cuda")
    args = (x, x) if cls == "DCNv2Pack" else (x,)
    with torch.no_grad():
        assert not m._fusable(x)
        y = m(*args)
        o1, o2, mk = torch.chunk(m.conv_offset(x), 3, dim=1)
        want = dcn.modulated_deform_conv(x, torch.cat((o1, o2), 1), torch.sigmoid(mk), m.weight, m.bias, stride, padding,
                                         1, 1, 8)
    Ho, Wo = (12 + 2 * padding - 3) // stride + 1, (14 + 2 * padding - 3) // stride + 1
    assert y.shape == (1, 64, Ho, Wo) and _err(y, want) < 1e-6


@pytest.mark.gpu
def test_mixed_dtype_call_keeps_the_fp32_path(cuda):
    """fp64 input with an fp32 offset is not an all-fp64 call: the shim converts to fp32 exactly as before."""
    from edvr_b200 import deform_conv_ext as ext
    from edvr_b200 import ops
    x, off, mask, w, b = (t.cuda() for t in _case(1, 64, 10, 12, 64, 3, 3, 1, 1, 1, 8, seed=31))
    out = torch.empty(1, 64, 10, 12, dtype=torch.float64, device="cuda")
    e = x.new_empty(0)
    ext.modulated_deform_conv_forward(x, w, b, e, off.float(), mask, out, e, 3, 3, 1, 1, 1, 1, 1, 1, 1, 8, True)
    want = ops.mdcn_forward(x.float(), off.float(), mask.float(), w.float(), b.float(), 1, 1, 1, 1, 8)
    assert torch.equal(out, want.double())


@pytest.mark.gpu
@pytest.mark.parametrize("C,dg,Cout,fp32_error", [(3, 1, 8, "C % 64"), (12, 3, 8, "C % 64"), (64, 8, 600, "Cout=600 > 512")])
def test_f64_has_no_channel_limits(cuda, C, dg, Cout, fp32_error):
    """Channel counts the fp32 tensor-core kernels reject work in fp64; the same calls in fp32 still raise."""
    from edvr_b200 import ops
    x, off, mask, w, b = _case(1, C, 7, 9, Cout, 3, 3, 1, 1, 1, dg, seed=C + Cout)
    ref = _tv(x, off, mask, w, b, 1, 1, 1, torch.zeros(1, Cout, 7, 9, dtype=torch.float64))[0]
    xc, oc, mc, wc, bc = (t.cuda() for t in (x, off, mask, w, b))
    got = ops.mdcn_forward(xc, oc, mc, wc, bc, 1, 1, 1, 1, dg)
    assert _err(got, ref) <= BAR
    with pytest.raises(RuntimeError, match=fp32_error):
        ops.mdcn_forward(xc.float(), oc.float(), mc.float(), wc.float(), bc.float(), 1, 1, 1, 1, dg)


# ---- 6. host-side validation (no GPU) --------------------------------------------------------------------------------
def test_f64_entries_validate_before_any_cuda_call():
    """Statuses of the fp64 entries for a null pointer (-5), a bad shape (-1), weight groups (-2) and a short workspace
    (-4), all decided on the host."""
    from edvr_b200 import _lib as L
    h = L.lib()
    p = L.ptr(torch.zeros(4, dtype=torch.float64))
    geo = (1, 12, 8, 8, 10, 3, 3)            # N, C, H, W, Cout, kh, kw: C % 64 != 0 is fine in fp64
    assert h.eb_mdcn_forward_f64(None, p, p, p, None, p, *geo, 1, 1, 1, 1, 3, None) == -5
    assert h.eb_mdcn_forward_f64(p, p, p, p, None, p, *geo, 0, 1, 1, 1, 3, None) == -1           # stride 0
    assert h.eb_mdcn_forward_f64(p, p, p, p, None, p, *geo, 1, 1, 1, 1, 5, None) == -1           # C % dg
    assert h.eb_mdcn_forward_f64(p, p, p, p, None, p, *geo, 1, 1, 1, 2, 3, None) == -2           # groups
    assert h.eb_dcn1_forward_f64(p, None, p, p, *geo, 1, 1, 1, 1, 1, 1, 1, 3, None) == -5
    assert h.eb_dcn1_forward_f64(p, p, p, p, *geo, 1, 1, 1, 1, 1, 1, 2, 3, None) == -2
    assert h.eb_dcn1_forward_f64(p, p, p, p, *geo, 1, 1, -1, 1, 1, 1, 1, 3, None) == -1          # pad -1

    # C*kh*kw or Cout beyond the 65535 tiles of 64 the grids can hold
    assert h.eb_mdcn_forward_f64(p, p, p, p, None, p, 1, 466034, 8, 8, 10, 3, 3, 1, 1, 1, 1, 1, None) == -2
    assert h.eb_mdcn_forward_f64(p, p, p, p, None, p, 1, 12, 8, 8, 65535 * 64 + 1, 3, 3, 1, 1, 1, 1, 3, None) == -2

    need = h.eb_mdcn_backward_f64_workspace(*geo, 1, 1, 1)
    assert need >= 12 * 9 * 64 * 8                                         # the column gradient of one image at least
    assert h.eb_dcn1_backward_input_f64_workspace(*geo, 1, 1, 1, 1, 1, 1) == need
    need_par = h.eb_dcn1_backward_parameters_f64_workspace(*geo, 1, 1, 1, 1, 1, 1)
    assert 10 * 12 * 9 * 8 <= need_par < need                              # one split of grad_weight partials, no gcol
    args = (p, p, p, p, p, p, p, p, p, p, *geo, 1, 1, 1)
    assert h.eb_mdcn_backward_f64(*args, 1, 3, p, need - 1, None) == -4
    assert b"workspace" in h.eb_last_error()
    assert h.eb_mdcn_backward_f64(*args, 2, 3, p, need, None) == -2
    assert h.eb_mdcn_backward_f64(p, p, None, *args[3:], 1, 3, p, need, None) == -5                # no mask
    v1 = (*geo, 1, 1, 1, 1, 1, 1)
    assert h.eb_dcn1_backward_input_f64(p, p, p, p, p, p, *v1, 1, 3, p, need - 1, None) == -4
    assert h.eb_dcn1_backward_input_f64(p, p, None, p, p, p, *v1, 1, 3, p, need, None) == -5
    assert h.eb_dcn1_backward_parameters_f64(p, p, p, p, 0.5, *v1, 1, 3, p, need_par - 1, None) == -4
    assert h.eb_dcn1_backward_parameters_f64(p, p, p, p, 0.5, *v1, 2, 3, p, need_par, None) == -2
    assert h.eb_dcn1_backward_parameters_f64(p, p, p, p, 0.5, 1, 12, 8, 8, 10, 3, 3, 1, 1, 1, 1, 0, 1, 1, 3, p, need,
                                             None) == -1                   # dilation 0
    # an empty batch is a no-op, pointers unused
    assert h.eb_mdcn_backward_f64(None, None, None, None, None, None, None, None, None, None, 0, 12, 8, 8, 10, 3, 3, 1, 1,
                                  1, 1, 3, None, 0, None) == 0
