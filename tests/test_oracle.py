"""CPU tests (-m "not gpu"): the oracle against every pin we have for this path.

The reference ships no golden vectors for dcn/EDVR (SURVEY §4), so the pins are
  (1) tests/golden/dcn_ref_cuda_*.npz — outputs of the UNMODIFIED reference CUDA extension on a B200
      (tools/first_light.py::sec_refext, built by oracle/build_ref.py);
  (2) torchvision.ops.deform_conv2d (same semantics except grad_offset at coordinate == -1);
  (3) tests/golden/edvr_ref_import_*.npz — the reference's own Python graph imported from
      /root/reference in the build container (oracle/make_golden.py).
"""
import glob
import os

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import dcn_oracle, edvr_ref

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _port_forward(sd, x, **kw):
    """edvr_ref.edvr_forward with the intra-op thread count of the recordings (oracle/make_golden.py): the CPU
    convolutions split their reductions by thread count, and bit-exact agreement needs the same split."""
    from oracle.make_golden import RECORDING_THREADS
    n = torch.get_num_threads()
    torch.set_num_threads(RECORDING_THREADS)
    try:
        return edvr_ref.edvr_forward(sd, x, **kw)
    finally:
        torch.set_num_threads(n)


def _rand_case(N, C, H, W, Cout, dg, seed=0, off_scale=3.0, k=3):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, C, H, W, generator=g)
    off = torch.randn(N, dg * 2 * k * k, H, W, generator=g) * off_scale
    mask = torch.sigmoid(torch.randn(N, dg * k * k, H, W, generator=g))
    w = torch.randn(Cout, C, k, k, generator=g) * 0.1
    b = torch.randn(Cout, generator=g)
    return x, off, mask, w, b


@pytest.mark.parametrize("shape", [(2, 16, 9, 11, 8, 4), (1, 8, 5, 7, 6, 1), (1, 32, 6, 6, 16, 8)])
def test_oracle_forward_backward_vs_torchvision(shape):
    from torchvision.ops import deform_conv2d
    N, C, H, W, Cout, dg = shape
    x, off, mask, w, b = _rand_case(*shape, seed=3)
    # keep sample coordinates away from exact integers: torchvision differs only at coord == -1
    for t in (x, off, mask, w, b):
        t.requires_grad_(True)
    y = deform_conv2d(x, off, w, b, stride=1, padding=1, dilation=1, mask=mask)
    go = torch.randn(y.shape, generator=torch.Generator().manual_seed(9))
    y.backward(go)
    d = lambda t: t.detach().numpy()
    yo = dcn_oracle.forward(d(x), d(off), d(mask), d(w), d(b), 1, 1, 1, 1, dg)
    assert rel_err(yo, y.detach())[0] < 1e-5
    grads = dcn_oracle.backward(d(x), d(off), d(mask), d(w), go.numpy(), True, 1, 1, 1, 1, dg)
    for name, got, ref in zip(("gx", "goff", "gmask", "gw", "gb"), grads, (x, off, mask, w, b)):
        assert rel_err(got, ref.grad)[0] < 2e-5, name


def test_oracle_stride_dilation_nobias_vs_torchvision():
    from torchvision.ops import deform_conv2d
    N, C, H, W, Cout, dg = 1, 8, 11, 13, 4, 2
    stride, pad, dil = 2, 2, 2
    Ho, Wo = dcn_oracle.out_hw(H, W, 3, 3, stride, pad, dil)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(N, C, H, W, generator=g)
    off = torch.randn(N, dg * 18, Ho, Wo, generator=g) * 2
    mask = torch.rand(N, dg * 9, Ho, Wo, generator=g)
    w = torch.randn(Cout, C, 3, 3, generator=g)
    y = deform_conv2d(x, off, w, None, stride=stride, padding=pad, dilation=dil, mask=mask)
    yo = dcn_oracle.forward(x.numpy(), off.numpy(), mask.numpy(), w.numpy(), None, stride, pad, dil, 1, dg)
    assert yo.shape == tuple(y.shape)
    assert rel_err(yo, y)[0] < 1e-5


def test_oracle_weight_groups_vs_torchvision():
    from torchvision.ops import deform_conv2d
    N, C, H, W, Cout, dg, groups = 1, 8, 6, 7, 6, 2, 2
    g = torch.Generator().manual_seed(6)
    x = torch.randn(N, C, H, W, generator=g)
    off = torch.randn(N, dg * 18, H, W, generator=g)
    mask = torch.rand(N, dg * 9, H, W, generator=g)
    w = torch.randn(Cout, C // groups, 3, 3, generator=g)
    y = deform_conv2d(x, off, w, None, padding=1, mask=mask)
    yo = dcn_oracle.forward(x.numpy(), off.numpy(), mask.numpy(), w.numpy(), None, 1, 1, 1, groups, dg)
    assert rel_err(yo, y)[0] < 1e-5


def test_oracle_minus_one_edge_follows_reference():
    """Zero offsets + padding 1 put every border tap exactly on coordinate -1: the reference returns
    grad_offset == 0 there (deform_conv_cuda_kernel.cu:747-750,531-535); torchvision does not."""
    N, C, H, W, Cout, dg = 1, 4, 5, 6, 3, 2
    x, off, mask, w, b = _rand_case(N, C, H, W, Cout, dg, seed=1, off_scale=0.0)
    go = torch.randn(N, Cout, H, W, generator=torch.Generator().manual_seed(2))
    gx, goff, gmask, gw, gb = dcn_oracle.backward(x.numpy(), off.numpy(), mask.numpy(), w.numpy(), go.numpy(),
                                                  True, 1, 1, 1, 1, dg)
    goff = goff.reshape(N, dg, 9, 2, H, W)
    # tap (0, *) at output row 0 samples h = -1 -> zero gradient for both dh and dw
    assert np.all(goff[:, :, 0:3, :, 0, :] == 0)
    assert np.all(goff[:, :, [0, 3, 6], :, :, 0] == 0)
    # interior taps do get gradient
    assert np.abs(goff[:, :, 4, :, 2, 2]).max() > 0


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "dcn_ref_cuda_*.npz"))))
def test_oracle_vs_reference_cuda_golden(path):
    z = np.load(path)
    N, C, H, W, Cout, dg, stride, pad, dil, groups = (int(v) for v in z["meta"])
    yo = dcn_oracle.forward(z["x"], z["offset"], z["mask"], z["weight"], z["bias"], stride, pad, dil, groups, dg)
    assert rel_err(yo, z["out"])[0] < 5e-6
    grads = dcn_oracle.backward(z["x"], z["offset"], z["mask"], z["weight"], z["grad_out"], True, stride, pad, dil,
                                groups, dg)
    for name, got in zip(("grad_x", "grad_offset", "grad_mask", "grad_weight", "grad_bias"), grads):
        assert rel_err(got, z[name])[0] < 5e-6, name


V1_CASES = [  # N, C, H, W, Cout, dg, (kh, kw), stride, padding, dilation
    (2, 8, 9, 11, 6, 2, (3, 3), (1, 1), (1, 1), (1, 1)),
    (1, 8, 12, 10, 4, 1, (3, 3), (2, 1), (1, 2), (1, 2)),
    (1, 16, 7, 9, 8, 4, (1, 3), (1, 2), (0, 1), (1, 1)),
]


@pytest.mark.parametrize("case", V1_CASES)
def test_oracle_v1_forward_backward_vs_torchvision(case):
    """DCNv1 (mask-less, bias-less, per-axis geometry, `scale` on grad_weight) against torchvision's autograd."""
    from torchvision.ops import deform_conv2d
    N, C, H, W, Cout, dg, k, s, p, d = case
    g = torch.Generator().manual_seed(13)
    Ho, Wo = ((sz + 2 * p[i] - (d[i] * (k[i] - 1) + 1)) // s[i] + 1 for i, sz in enumerate((H, W)))
    x = torch.randn(N, C, H, W, generator=g, requires_grad=True)
    off = (torch.randn(N, dg * 2 * k[0] * k[1], Ho, Wo, generator=g) * 2).requires_grad_(True)
    w = (torch.randn(Cout, C, *k, generator=g) * 0.1).requires_grad_(True)
    y = deform_conv2d(x, off, w, None, stride=s, padding=p, dilation=d)
    go = torch.randn(y.shape, generator=g)
    y.backward(go)
    dn = lambda t: t.detach().numpy()
    yo = dcn_oracle.forward_v1(dn(x), dn(off), dn(w), s, p, d, 1, dg)
    assert yo.shape == tuple(y.shape) and rel_err(yo, y.detach())[0] < 1e-5
    gx, goff, gw = dcn_oracle.backward_v1(dn(x), dn(off), dn(w), go.numpy(), s, p, d, 1, dg, scale=0.25)
    assert rel_err(gx, x.grad)[0] < 2e-5 and rel_err(goff, off.grad)[0] < 2e-5
    assert rel_err(gw, 0.25 * w.grad)[0] < 2e-5


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "dcn1_ref_cuda_*.npz"))))
def test_oracle_v1_vs_reference_cuda_golden(path):
    """Pins the DCNv1 oracle on outputs of the unmodified reference CUDA extension (tools/first_light.py refext_v1)."""
    z = np.load(path)
    N, C, H, W, Cout, dg, kh, kw, sh, sw, ph, pw, dh, dw = (int(v) for v in z["meta"])
    s, p, d = (sh, sw), (ph, pw), (dh, dw)
    yo = dcn_oracle.forward_v1(z["x"], z["offset"], z["weight"], s, p, d, 1, dg)
    assert rel_err(yo, z["out"])[0] < 1e-5
    gx, goff, gw = dcn_oracle.backward_v1(z["x"], z["offset"], z["weight"], z["grad_out"], s, p, d, 1, dg,
                                          scale=float(z["scale"]))
    for name, got in (("grad_x", gx), ("grad_offset", goff), ("grad_weight", gw)):
        assert rel_err(got, z[name])[0] < 2e-5, name


def test_oracle_rejects_bad_shapes():
    x = np.zeros((1, 6, 4, 4), np.float32)
    with pytest.raises(ValueError):
        dcn_oracle.forward(x, np.zeros((1, 18 * 4, 4, 4), np.float32), np.zeros((1, 9 * 4, 4, 4), np.float32),
                           np.zeros((4, 6, 3, 3), np.float32), None, 1, 1, 1, 1, 4)   # 6 % 4 != 0


def test_oracle_empty_batch():
    x = np.zeros((0, 4, 4, 4), np.float32)
    y = dcn_oracle.forward(x, np.zeros((0, 18, 4, 4), np.float32), np.zeros((0, 9, 4, 4), np.float32),
                           np.zeros((2, 4, 3, 3), np.float32), None, 1, 1, 1, 1, 1)
    assert y.shape == (0, 2, 4, 4)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "edvr_ref_import_*.npz"))))
def test_edvr_port_matches_reference_import_golden(path):
    """The functional port reproduces, bit for bit, outputs recorded from the imported reference graph."""
    z = np.load(path, allow_pickle=True)
    kw = z["kwargs"].item()
    sd = edvr_ref.make_state_dict(**{k: v for k, v in kw.items() if k not in ("center_frame_idx",)}, seed=int(z["seed"]))
    x = torch.from_numpy(z["x"])
    y = _port_forward(sd, x, hr_in=kw.get("hr_in", False))
    assert torch.equal(y, torch.from_numpy(z["y"]))


def test_edvr_port_matches_reference_import_live():
    """The reference graph imported unchanged (oracle/make_golden_live.py) on the weights of make_state_dict and a seeded
    input: bit-identical output, same state_dict keys (tests/golden/ref_live.npz, ref_host.json)."""
    import json
    with open(os.path.join(GOLDEN, "ref_host.json")) as f:
        ref = json.load(f)["port_edvr"]
    z = np.load(os.path.join(GOLDEN, "ref_live.npz"))
    sd = edvr_ref.make_state_dict(**ref["kwargs"], seed=ref["seed"])
    x = torch.from_numpy(z["edvr_x"])
    assert torch.equal(torch.from_numpy(z["edvr_y"]), _port_forward(sd, x))
    assert sorted(sd) == ref["state_dict_keys"]


# ---- frame staging either side of the network (SURVEY §8 f2): oracle/img_ref.py ---------------------------------------
GOLDEN_IMG = os.path.join(GOLDEN, "img_ref_import.npz")


def test_img_oracle_matches_reference_import_golden_bit_exact():
    """oracle/img_ref.py against tests/golden/img_ref_import.npz, recorded from the UNMODIFIED basicsr.utils.img_util /
    data_util arithmetic (oracle/make_golden_img.py): byte and fp32-bit equality."""
    from oracle import img_ref
    z = np.load(GOLDEN_IMG)
    x = img_ref.frames_to_tensor(z["frames"])
    assert x.dtype == np.float32 and np.array_equal(x.view(np.uint32), z["x"].view(np.uint32))
    assert np.array_equal(img_ref.tensor2img(z["out"]), z["y"])
    assert np.array_equal(img_ref.tensor2img(z["out"], rgb2bgr=False), z["y_rgb"])
    assert np.array_equal(img_ref.tensor2img(z["out"][:, :1]), z["gray"]) and z["gray"].ndim == 2
    assert np.array_equal(img_ref.tensor2img(z["out"] * 2 - 1, min_max=(-1, 1)), z["y_pm1"])
    # every byte survives the round trip frames -> [0, 1] floats -> bytes
    ramp = np.arange(256, dtype=np.uint8).reshape(1, 16, 16, 1).repeat(3, axis=3)
    assert np.array_equal(img_ref.tensor2img(img_ref.frames_to_tensor(ramp)[0]), ramp[0])


def test_img_oracle_matches_live_reference_import():
    """The reference's img2tensor / tensor2img on seeded frames and outputs (tests/golden/ref_live.npz,
    oracle/make_golden_live.py)."""
    from oracle import img_ref
    z = np.load(os.path.join(GOLDEN, "ref_live.npz"))
    frames, out = z["img_frames"], z["img_out"]
    assert np.array_equal(img_ref.frames_to_tensor(frames).view(np.uint32), z["img_x"].view(np.uint32))
    assert np.array_equal(img_ref.tensor2img(out), z["img_y"])
    assert np.array_equal(img_ref.tensor2img(out[0, 0]), z["img_y00"]) and z["img_y00"].ndim == 2
