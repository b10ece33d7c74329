"""Role-level cycle counters of conv_igemm2 (eb_conv2d_stats) + isolated timing of one conv call."""
import ctypes
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from edvr_b200 import _lib as L, ops  # noqa: E402

NAMES = ["mma_total", "mma_wait_acc", "mma_wait_a", "mma_wait_w", "a_total", "a_wait_empty", "w_total",
         "w_wait_empty", "epi_total", "epi_wait_acc", "tiles", "e_tmem", "e_p1", "e_bar", "e_p2"]


def time_it(fn, iters=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def conv_case(N, H, W, cin, cout, k, res32=False, label=""):
    x = ops.nchw_to_nhwc(torch.randn(N, cin, H, W, device="cuda"))
    w = torch.randn(cout, cin, k, k, device="cuda") / (cin * k * k) ** 0.5
    pc = ops.pack_conv(w, torch.zeros(cout, device="cuda"))
    out = ops.new_act(N, H, W, cout)
    stream = torch.zeros(N, H, W, cout, device="cuda") if res32 else None
    fl = 2.0 * N * H * W * cout * cin * k * k
    for variant in ("v2", "v1"):
        os.environ["EDVR_B200_CONV_V1"] = "1" if variant == "v1" else "0"
        os.environ["EDVR_B200_CONV_V2"] = "0" if variant == "v1" else "1"
        ms = time_it(lambda: ops.conv2d(pc, [x], out16=out, act=ops.ACT_RELU, res32=stream, out32=stream))
        print(f"{label} {variant}: N={N} {H}x{W} {cin}->{cout} k{k} res32={res32}: {ms*1e3:.1f} us  {fl/ms/1e9:.0f} TFLOP/s", flush=True)
    os.environ["EDVR_B200_CONV_V1"] = "0"
    if pc.BN == 128:
      for dbg in ([0, 1, 2, 6] if label.startswith("trunk conv1") else [0]):
        os.environ["EDVR_B200_DBG"] = str(dbg)
        stats = torch.zeros(148 * 16, dtype=torch.int64, device="cuda")
        arr = (L.Src * 1)(ops._src(x))
        e = ops._epi(pc.b, ops.ACT_RELU, out, stream, None, stream)
        L.check(L.lib().eb_conv2d_stats(arr, 1, N, H, W, k, L.ptr(pc.w), pc.BN, pc.n_tiles, ctypes.byref(e),
                                        L.ptr(stats), L.stream_ptr()))
        torch.cuda.synchronize()
        st = stats.view(148, 16).double()
        used = st[:, 10] > 0
        m = st[used].mean(0)
        tiles = float(m[10])
        print(f"   dbg={dbg} cycles/tile: mma_total {m[0]/tiles:.0f}  wait_acc {m[1]/tiles:.0f} wait_a {m[2]/tiles:.0f} wait_w {m[3]/tiles:.0f} | "
              f"A idle {m[5]/tiles:.0f} of {m[4]/tiles:.0f} | W idle {m[7]/tiles:.0f} | epi wait {m[9]/tiles:.0f} of {m[8]/tiles:.0f} | "
              f"epi: tmem {m[11]/tiles:.0f} p1 {m[12]/tiles:.0f} bar {m[13]/tiles:.0f} p2 {m[14]/tiles:.0f}", flush=True)


if __name__ == "__main__":
    conv_case(4, 180, 320, 128, 128, 3, label="trunk conv1")
    conv_case(4, 180, 320, 128, 128, 3, res32=True, label="trunk conv2")
    conv_case(28, 180, 320, 128, 128, 3, label="feature extraction")
    conv_case(28, 180, 320, 256, 128, 3, label="pcd cat conv")
    conv_case(28, 180, 320, 128, 256, 3, label="conv_offset-like")
    conv_case(4, 180, 320, 896, 256, 1, label="tsa fuse 1x1")
    conv_case(4, 720, 1280, 64, 64, 3, label="conv_hr")
    conv_case(4, 360, 640, 128, 256, 3, label="upconv2")
