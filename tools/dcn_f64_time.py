"""Device-event timing of the double-precision DCNv2 operator (eb_mdcn_forward_f64 / eb_mdcn_backward_f64).

Prints the GPU name and power limit, then per shape the time per call and the achieved fp64 rate.  FLOPs come from the
shapes: the forward GEMM is 2 * N*Ho*Wo * C*kh*kw * Cout (EDVR-L L1, 1x128x180x320 -> 128, 3x3: ~17.0 GFLOP); the backward
runs two GEMMs of that size (column gradient and weight gradient).  The bilinear gathers are not counted.

    python tools/dcn_f64_time.py [--iters 20]
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from edvr_b200 import _lib as L  # noqa: E402

SHAPES = [   # name, N, C, H, W, Cout, dg
    ("edvr_l_L1", 1, 128, 180, 320, 128, 8),
    ("small", 2, 64, 48, 64, 64, 8),
]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # report what is known rather than nothing
        q = f"{torch.cuda.get_device_name(0)}, power limit unknown ({e!r})"
    return q


def time_call(fn, iters):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dcn_f64_time.py needs a CUDA device")
    print(f"gpu: {card()}")
    h = L.lib()
    g = torch.Generator(device="cuda").manual_seed(0)
    for name, N, C, H, W, Cout, dg in SHAPES:
        kh = kw = 3
        K = kh * kw
        dev = dict(device="cuda", dtype=torch.float64)
        x = torch.randn(N, C, H, W, generator=g, **dev)
        off = torch.randn(N, dg * 2 * K, H, W, generator=g, **dev) * 2
        mask = torch.rand(N, dg * K, H, W, generator=g, **dev)
        w = torch.randn(Cout, C, kh, kw, generator=g, **dev) / (C * K) ** 0.5
        b = torch.randn(Cout, generator=g, **dev)
        out = torch.empty(N, Cout, H, W, **dev)
        go = torch.randn(N, Cout, H, W, generator=g, **dev)
        gx, goff, gm = torch.empty_like(x), torch.empty_like(off), torch.empty_like(mask)
        gw, gb = torch.zeros_like(w), torch.zeros_like(b)
        need = h.eb_mdcn_backward_f64_workspace(N, C, H, W, Cout, kh, kw, 1, 1, 1)
        ws = torch.empty(need, dtype=torch.uint8, device="cuda")
        st = L.stream_ptr()

        def fwd():
            L.check(h.eb_mdcn_forward_f64(L.ptr(x), L.ptr(off), L.ptr(mask), L.ptr(w), L.ptr(b), L.ptr(out), N, C, H, W,
                                          Cout, kh, kw, 1, 1, 1, 1, dg, st), "eb_mdcn_forward_f64")

        def bwd():
            L.check(h.eb_mdcn_backward_f64(L.ptr(x), L.ptr(off), L.ptr(mask), L.ptr(w), L.ptr(go), L.ptr(gx), L.ptr(goff),
                                           L.ptr(gm), L.ptr(gw), L.ptr(gb), N, C, H, W, Cout, kh, kw, 1, 1, 1, 1, dg,
                                           L.ptr(ws), ws.numel(), st), "eb_mdcn_backward_f64")

        flops = 2.0 * N * H * W * C * K * Cout
        tf, tb = time_call(fwd, args.iters), time_call(bwd, args.iters)
        print(f"{name} {N}x{C}x{H}x{W} dg{dg} Cout{Cout} 3x3: forward {tf * 1e3:.3f} ms ({flops / 1e9:.1f} GFLOP, "
              f"{flops / tf / 1e12:.2f} TFLOP/s fp64); backward {tb * 1e3:.3f} ms ({2 * flops / 1e9:.1f} GFLOP, "
              f"{2 * flops / tb / 1e12:.2f} TFLOP/s fp64); workspace {need / 2**20:.0f} MiB")


if __name__ == "__main__":
    main()
