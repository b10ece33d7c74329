"""Launch one DCN site (ops.DcnSite) a few times on one shape: ncu target.
    python tools/one_site.py N H W C dg sigma [iters]      (mode: EDVR_B200_DCN_SITE=pair|fused|split)"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from edvr_b200 import ops  # noqa: E402
from dcn_sweep import site_weights  # noqa: E402

a = sys.argv[1:]
N, H, W, C, dg = (int(v) for v in (a[:5] if len(a) >= 5 else (4, 180, 320, 128, 8)))
sigma = float(a[5]) if len(a) > 5 else 0.02
iters = int(a[6]) if len(a) > 6 else 3
wo, bo, w, b = site_weights(C, dg, sigma, torch.Generator().manual_seed(1))
g = torch.Generator(device="cuda").manual_seed(0)
x = ops.nchw_to_nhwc(torch.randn(N, C, H, W, device="cuda", generator=g))
feat = ops.nchw_to_nhwc(torch.randn(N, C, H, W, device="cuda", generator=g))
out = ops.new_act(N, H, W, C)
site = ops.DcnSite(wo, bo, w, b, dg)
for _ in range(iters):
    site(x, feat, out)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(iters):
    site(x, feat, out)
e1.record()
torch.cuda.synchronize()
print(f"site {site.mode} N={N} {H}x{W} C={C} sigma={sigma}: {e0.elapsed_time(e1) * 1e3 / iters:.1f} us, checksum {float(out.t.float().abs().mean()):.6f}")
