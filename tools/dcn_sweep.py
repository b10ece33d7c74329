"""DCN site (conv_offset -> DCN) at several offset magnitudes: parity vs the C oracle on a small shape and device time
of the site's launches at full size.  `sigma` is the standard deviation of the sampling offsets in pixels (iid per pixel,
group and tap: the worst case for locality; trained EDVR offsets are smoother).

    python tools/dcn_sweep.py [--n 28] [--sigmas 0.02,3,10] [--json gpurun_out/dcn_sweep.json]
"""
import argparse
import json
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from edvr_b200 import ops  # noqa: E402


def site_weights(C, dg, sigma, gen, device="cuda"):
    """conv_offset weights such that the offsets come out ~ N(0, sigma^2) for unit-variance input features."""
    wo = torch.randn(dg * 27, C, 3, 3, generator=gen) / (C * 9) ** 0.5
    wo[:dg * 18] *= sigma                       # offset rows; the mask logits stay O(1)
    bo = torch.randn(dg * 27, generator=gen) * 0.1
    w = (torch.rand(C, C, 3, 3, generator=gen) * 2 - 1) / (C * 9) ** 0.5
    b = torch.randn(C, generator=gen) * 0.1
    return [t.to(device) for t in (wo, bo, w, b)]


def parity(sigma, N=2, C=128, H=18, W=23, dg=8):
    from oracle import dcn_oracle        # checker only (tools/ is test infrastructure)
    gen = torch.Generator().manual_seed(2)
    x = torch.randn(N, C, H, W, generator=gen)
    feat = torch.randn(N, C, H, W, generator=gen)
    wo, bo, w, b = site_weights(C, dg, sigma, gen, "cpu")
    raw = F.conv2d(feat.half().double(), wo.half().double(), bo.double(), padding=1).float()
    off, mask = raw[:, :dg * 18].contiguous(), torch.sigmoid(raw[:, dg * 18:]).contiguous()
    ref = torch.from_numpy(dcn_oracle.forward(x.numpy(), off.numpy(), mask.numpy(), w.numpy(), b.numpy(), 1, 1, 1, 1, dg))
    out = ops.new_act(N, H, W, C)
    site = ops.DcnSite(wo.cuda(), bo.cuda(), w.cuda(), b.cuda(), dg)
    site(ops.nchw_to_nhwc(x.cuda()), ops.nchw_to_nhwc(feat.cuda()), out)
    got = ops.nhwc_to_nchw(out).cpu()
    d = (got - ref).double()
    return {"sigma": sigma, "shape": [N, C, H, W, dg], "offset_absmean": float(off.abs().mean()),
            "max_rel": float(d.abs().max() / ref.abs().max()), "l2_rel": float(d.norm() / ref.double().norm())}


def timing(sigma, N, H=180, W=320, C=128, dg=8, iters=5):
    gen = torch.Generator().manual_seed(1)
    wo, bo, w, b = site_weights(C, dg, sigma, gen)
    g = torch.Generator(device="cuda").manual_seed(0)
    x = ops.nchw_to_nhwc(torch.randn(N, C, H, W, device="cuda", generator=g))
    feat = ops.nchw_to_nhwc(torch.randn(N, C, H, W, device="cuda", generator=g))
    out = ops.new_act(N, H, W, C)
    site = ops.DcnSite(wo, bo, w, b, dg)
    for _ in range(2):
        site(x, feat, out)
    torch.cuda.synchronize()
    ops.PROFILE = []
    for _ in range(iters):
        site(x, feat, out)
    torch.cuda.synchronize()
    recs, ops.PROFILE = ops.PROFILE, None
    agg = {}
    for name, flops, e0, e1, _d in recs:
        a = agg.setdefault(name, [0.0, 0.0])
        a[0] += e0.elapsed_time(e1) * 1e3 / iters
        a[1] += flops / iters
    res = {"sigma": sigma, "N": N, "HxW": f"{H}x{W}"}
    for k, (us, fl) in agg.items():
        res[k + "_us"] = round(us, 1)
        res[k + "_tflops"] = round(fl / us / 1e6, 1)
    res["site_us"] = round(sum(v[0] for v in agg.values()), 1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", default="28,4")
    ap.add_argument("--sigmas", default="0.02,3,10")
    ap.add_argument("--json", default=os.path.join(ROOT, "gpurun_out", "dcn_sweep.json"))
    ap.add_argument("--modes", default="pair,fused", help="ops.DcnSite modes to compare")
    a = ap.parse_args()
    res = {"parity": [], "timing": []}
    for mode in a.modes.split(","):
        os.environ["EDVR_B200_DCN_SITE"] = mode
        for s in [float(v) for v in a.sigmas.split(",")]:
            for shape in ((2, 128, 18, 23, 8), (1, 64, 16, 24, 8), (3, 64, 21, 9, 4)):
                r = dict(parity(s, *shape), mode=mode)
                print("parity", r, flush=True)
                res["parity"].append(r)
    for n in [int(v) for v in a.n.split(",")]:
        for mode in a.modes.split(","):
            os.environ["EDVR_B200_DCN_SITE"] = mode
            for s in [float(v) for v in a.sigmas.split(",")]:
                r = dict(timing(s, n), mode=mode)
                print("timing", r, flush=True)
                res["timing"].append(r)
    os.makedirs(os.path.dirname(a.json), exist_ok=True)
    with open(a.json, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
