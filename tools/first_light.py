"""GPU bring-up script (run under gpurun): each section runs in its own subprocess so that a
trap in one kernel cannot poison the others.  Results are printed and saved to gpurun_out/.

    python tools/first_light.py            # all sections
    python tools/first_light.py --section selftest
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "gpurun_out")
os.makedirs(OUT, exist_ok=True)


def rel(a, b):
    import torch
    a, b = a.float(), b.float()
    return dict(max_abs=float((a - b).abs().max()), ref_max=float(b.abs().max()),
                rel_max=float((a - b).abs().max() / b.abs().max().clamp_min(1e-20)),
                rel_l2=float((a - b).norm() / b.norm().clamp_min(1e-20)))


def sec_selftest():
    import torch
    from edvr_b200 import _lib as L
    res = {}
    for (N, K) in [(128, 64), (128, 128), (64, 32), (256, 16), (96, 64)]:
        torch.manual_seed(0)
        A = torch.randn(128, K, device="cuda").half()
        B = torch.randn(N, K, device="cuda").half()
        ref = A.float() @ B.float().t()
        for variant in (0,):   # other variants probe wrong conventions (they fault)
            D = torch.full((128, N), float("nan"), device="cuda")
            rc = L.lib().eb_selftest_umma(L.ptr(A), L.ptr(B), L.ptr(D), N, K, variant, L.stream_ptr())
            torch.cuda.synchronize()
            r = rel(D, ref) if rc == 0 else {"rc": rc}
            res[f"N{N}_K{K}_v{variant}"] = r
            print(f"selftest N={N} K={K} variant={variant}: {r}", flush=True)
    return res


def sec_conv():
    import torch
    import torch.nn.functional as F
    from edvr_b200 import ops
    res = {}
    torch.manual_seed(1)

    def run(name, N, H, W, cins, cout, k, act=ops.ACT_NONE, res16=False, out_mode=ops.OUT_SAME, maps=None):
        xs = [torch.randn(N if (maps is None or maps[i] is None) else maps[i][4], c, H, W, device="cuda")
              for i, c in enumerate(cins)]
        w = torch.randn(cout, sum(cins), k, k, device="cuda") * (1.0 / (sum(cins) * k * k) ** 0.5)
        b = torch.randn(cout, device="cuda") * 0.1
        pc = ops.pack_conv(w, b)
        views = [ops.nchw_to_nhwc(x) for x in xs]
        # reference on the fp16-rounded operands, fp32 math
        xr = []
        for i, x in enumerate(xs):
            xh = x.half().float()
            if maps is not None and maps[i] is not None:
                div, mul, keep, add, _ = maps[i]
                idx = torch.tensor([(n // div) * mul + (n % div) * keep + add for n in range(N)], device="cuda")
                xh = xh[idx]
            xr.append(xh)
        wr = w.half().float()
        y = F.conv2d(torch.cat(xr, 1), wr, b, 1, k // 2)
        if act == ops.ACT_RELU:
            y = F.relu(y)
        elif act == ops.ACT_LRELU:
            y = F.leaky_relu(y, 0.1)
        r16 = None
        if res16:
            rt = torch.randn(N, cout, H, W, device="cuda")
            r16 = ops.nchw_to_nhwc(rt)
            y = y + rt.half().float()
        if out_mode == ops.OUT_PIXSHUF2:
            y = F.pixel_shuffle(y, 2)
            out = ops.new_act(N, 2 * H, 2 * W, cout // 4)
        elif out_mode == ops.OUT_STRIDE2:
            y = y[:, :, ::2, ::2]
            out = ops.new_act(N, (H + 1) // 2, (W + 1) // 2, cout)
        else:
            out = ops.new_act(N, H, W, cout)
        out.t.fill_(float("nan"))
        sm = None if maps is None else [None if m is None else m[:4] for m in maps]
        ops.conv2d(pc, views, out16=out, act=act, res16=r16, out_mode=out_mode, src_maps=sm, N=N)
        torch.cuda.synchronize()
        got = ops.nhwc_to_nchw(out)
        torch.cuda.synchronize()
        r = rel(got, y)
        r["nan"] = int(torch.isnan(got).sum())
        res[name] = r
        print(f"conv {name}: {r}", flush=True)

    run("3x3_c64_o64_small", 1, 16, 16, [64], 64, 3)
    run("3x3_c64_o64_ragged", 2, 21, 37, [64], 64, 3)
    run("3x3_c128_o128", 2, 45, 80, [128], 128, 3, act=ops.ACT_LRELU)
    run("1x1_c128_o128", 1, 33, 50, [128], 128, 1, act=ops.ACT_RELU)
    run("3x3_cat_128_128_o128_res", 3, 24, 40, [128, 128], 128, 3, res16=True)
    run("3x3_bcast_src1", 4, 20, 24, [64, 64], 64, 3, maps=[None, (2, 2, 0, 1, 4)])
    run("3x3_c128_o512_pixshuf", 1, 18, 20, [128], 512, 3, act=ops.ACT_LRELU, out_mode=ops.OUT_PIXSHUF2)
    run("3x3_c64_o64_stride2", 2, 22, 30, [64], 64, 3, act=ops.ACT_LRELU, out_mode=ops.OUT_STRIDE2)
    run("1x1_c896_o256", 1, 20, 32, [896], 256, 1, act=ops.ACT_LRELU)
    run("3x3_c128_o96", 1, 20, 20, [128], 96, 3)
    return res


def _dcn_inputs(N, C, H, W, Cout, dg, seed=0, off_scale=2.0):
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, C, H, W, generator=g)
    off = torch.randn(N, dg * 18, H, W, generator=g) * off_scale
    mask = torch.sigmoid(torch.randn(N, dg * 9, H, W, generator=g))
    w = (torch.rand(Cout, C, 3, 3, generator=g) * 2 - 1) / (C * 9) ** 0.5
    b = torch.randn(Cout, generator=g) * 0.1
    go = torch.randn(N, Cout, H, W, generator=g)
    return x, off, mask, w, b, go


def sec_dcn():
    import numpy as np
    import torch
    from edvr_b200 import ops
    from oracle import dcn_oracle
    res = {}
    for name, (N, C, H, W, Cout, dg) in {"cfg1_64": (1, 64, 64, 64, 64, 8), "c128_ragged": (2, 128, 19, 27, 128, 8),
                                          "c64_dg4": (1, 64, 9, 11, 32, 4)}.items():
        x, off, mask, w, b, _ = _dcn_inputs(N, C, H, W, Cout, dg)
        ref = torch.from_numpy(dcn_oracle.forward(x.numpy(), off.numpy(), mask.numpy(), w.numpy(), b.numpy(),
                                                  1, 1, 1, 1, dg))
        got = ops.mdcn_forward(x.cuda(), off.cuda(), mask.cuda(), w.cuda(), b.cuda(), 1, 1, 1, 1, dg)
        torch.cuda.synchronize()
        r = rel(got.cpu(), ref)
        r["nan"] = int(torch.isnan(got).sum())
        res[name] = r
        print(f"dcn {name}: {r}", flush=True)
    return res


def _ref_fns():
    """(forward, backward) wrappers over the UNMODIFIED reference CUDA extension (oracle/_ref)."""
    import torch
    from oracle import build_ref
    ext = build_ref.load_ref()

    def fwd(x, off, mask, w, b, stride, pad, dil, groups, dg):
        N, C, H, W = x.shape
        Cout, _, kh, kw = w.shape
        Ho = (H + 2 * pad - (dil * (kh - 1) + 1)) // stride + 1
        Wo = (W + 2 * pad - (dil * (kw - 1) + 1)) // stride + 1
        out = x.new_empty(N, Cout, Ho, Wo)
        bb = b if b is not None else x.new_empty(1)
        ext.modulated_deform_conv_forward(x, w, bb, x.new_empty(0), off, mask, out, x.new_empty(0), kh, kw, stride,
                                          stride, pad, pad, dil, dil, groups, dg, b is not None)
        return out

    def bwd(x, off, mask, w, b, go, stride, pad, dil, groups, dg):
        kh, kw = w.shape[2:]
        gx, goff, gm, gw = (torch.zeros_like(t) for t in (x, off, mask, w))
        gb = torch.zeros_like(b) if b is not None else x.new_zeros(1)
        bb = b if b is not None else x.new_empty(1)
        ext.modulated_deform_conv_backward(x, w, bb, x.new_empty(0), off, mask, x.new_empty(0), gx, gw, gb, goff, gm,
                                           go.contiguous(), kh, kw, stride, stride, pad, pad, dil, dil, groups, dg,
                                           b is not None)
        return gx, goff, gm, gw, (gb if b is not None else None)

    return fwd, bwd


def sec_refext():
    """Run the reference CUDA ext: compare with the C oracle, our kernel, and emit golden vectors."""
    import numpy as np
    import torch
    from edvr_b200 import ops
    from oracle import dcn_oracle
    fwd, bwd = _ref_fns()
    res = {}
    gold_dir = os.path.join(OUT, "golden")
    os.makedirs(gold_dir, exist_ok=True)
    cases = {"g_c64_dg8": (1, 64, 12, 14, 64, 8, 2.0), "g_c128_dg8": (2, 128, 10, 9, 128, 8, 3.0),
             "g_c64_dg4_zero_off": (1, 64, 8, 8, 32, 4, 0.0)}
    for name, (N, C, H, W, Cout, dg, osc) in cases.items():
        x, off, mask, w, b, go = _dcn_inputs(N, C, H, W, Cout, dg, seed=7, off_scale=osc)
        xc, oc, mc, wc, bc, gc = (t.cuda() for t in (x, off, mask, w, b, go))
        y = fwd(xc, oc, mc, wc, bc, 1, 1, 1, 1, dg)
        grads = bwd(xc, oc, mc, wc, bc, gc, 1, 1, 1, 1, dg)
        torch.cuda.synchronize()
        yo = torch.from_numpy(dcn_oracle.forward(x.numpy(), off.numpy(), mask.numpy(), w.numpy(), b.numpy(), 1, 1, 1, 1, dg))
        go_ = dcn_oracle.backward(x.numpy(), off.numpy(), mask.numpy(), w.numpy(), go.numpy(), True, 1, 1, 1, 1, dg)
        r = {"fwd_oracle_vs_ref": rel(yo, y.cpu())}
        for nm, a, bb in zip(("gx", "goff", "gmask", "gw", "gb"), go_, grads):
            r[f"{nm}_oracle_vs_ref"] = rel(torch.from_numpy(a), bb.cpu())
        ours = ops.mdcn_forward(xc, oc, mc, wc, bc, 1, 1, 1, 1, dg)
        torch.cuda.synchronize()
        r["fwd_ours_vs_ref"] = rel(ours.cpu(), y.cpu())
        res[name] = r
        print(f"refext {name}: {json.dumps(r)}", flush=True)
        np.savez_compressed(os.path.join(gold_dir, f"dcn_ref_cuda_{name}.npz"),
                            x=x.numpy(), offset=off.numpy(), mask=mask.numpy(), weight=w.numpy(), bias=b.numpy(),
                            grad_out=go.numpy(), out=y.cpu().numpy(), grad_x=grads[0].cpu().numpy(),
                            grad_offset=grads[1].cpu().numpy(), grad_mask=grads[2].cpu().numpy(),
                            grad_weight=grads[3].cpu().numpy(), grad_bias=grads[4].cpu().numpy(),
                            meta=np.array([N, C, H, W, Cout, dg, 1, 1, 1, 1]))
    return res


V1_CASES = {  # name: N, C, H, W, Cout, dg, (kh, kw), stride, padding, dilation, offset scale
    "v1_c64_dg8": (2, 64, 12, 14, 64, 8, (3, 3), (1, 1), (1, 1), (1, 1), 2.0),
    "v1_c64_dg1_aniso": (2, 64, 15, 13, 32, 1, (3, 3), (2, 1), (1, 2), (1, 2), 3.0),
    "v1_c128_dg4_k1x3": (1, 128, 9, 11, 128, 4, (1, 3), (1, 1), (0, 1), (1, 1), 1.5),
}


def _v1_inputs(N, C, H, W, Cout, dg, k, stride, pad, dil, osc, seed=11):
    import torch
    g = torch.Generator().manual_seed(seed)
    Ho = (H + 2 * pad[0] - (dil[0] * (k[0] - 1) + 1)) // stride[0] + 1
    Wo = (W + 2 * pad[1] - (dil[1] * (k[1] - 1) + 1)) // stride[1] + 1
    x = torch.randn(N, C, H, W, generator=g)
    off = torch.randn(N, dg * 2 * k[0] * k[1], Ho, Wo, generator=g) * osc
    w = (torch.rand(Cout, C, *k, generator=g) * 2 - 1) / (C * k[0] * k[1]) ** 0.5
    go = torch.randn(N, Cout, Ho, Wo, generator=g)
    return x, off, w, go


def sec_refext_v1():
    """DCNv1 entry points of the reference CUDA ext: compare with the C oracle and our kernels, emit golden vectors."""
    import numpy as np
    import torch
    from edvr_b200 import deform_conv_ext as ours
    from oracle import build_ref, dcn_oracle
    ext = build_ref.load_ref()
    res = {}
    gold_dir = os.path.join(OUT, "golden")
    os.makedirs(gold_dir, exist_ok=True)

    def run(mod, x, off, w, go, k, s, p, d, dg, scale, is_ref=False):
        # On current torch the reference's v1 host code only runs for some im2col_step values: forward re-views `columns`
        # inside its batch loop (needs a single iteration, step == N; deform_conv_cuda.cpp:222-226), backward_parameters
        # views a zeros_like() of a transposed tensor (needs step == 1; :425-434).  The result does not depend on the
        # step, so the reference is called with whichever step it accepts.
        N = x.shape[0]
        geom = (k[1], k[0], s[1], s[0], p[1], p[0], d[1], d[0], 1, dg)
        e = lambda: x.new_empty(0)

        def call(fn, *args):
            steps = (N, 1) if is_ref else (N,)
            for i, st in enumerate(steps):
                try:
                    return fn(*args, st)
                except RuntimeError:
                    if i == len(steps) - 1:
                        raise

        out = x.new_empty(go.shape)
        call(mod.deform_conv_forward, x, w, off, out, e(), e(), *geom)
        gx, goff, gw = torch.zeros_like(x), torch.zeros_like(off), torch.zeros_like(w)
        call(mod.deform_conv_backward_input, x, off, go, gx, goff, w, e(), *geom)
        try:
            mod.deform_conv_backward_parameters(x, off, go, gw, e(), e(), *geom, scale, N)
        except RuntimeError:
            if not is_ref:
                raise
            gw.zero_()
            mod.deform_conv_backward_parameters(x, off, go, gw, e(), e(), *geom, scale, 1)
        torch.cuda.synchronize()
        return out, gx, goff, gw

    for name, (N, C, H, W, Cout, dg, k, s, p, d, osc) in V1_CASES.items():
        x, off, w, go = _v1_inputs(N, C, H, W, Cout, dg, k, s, p, d, osc)
        cu = [t.cuda() for t in (x, off, w, go)]
        ref = run(ext, *cu, k, s, p, d, dg, 0.5, is_ref=True)
        yo = dcn_oracle.forward_v1(x.numpy(), off.numpy(), w.numpy(), s, p, d, 1, dg)
        go_ = dcn_oracle.backward_v1(x.numpy(), off.numpy(), w.numpy(), go.numpy(), s, p, d, 1, dg, scale=0.5)
        r = {"fwd_oracle_vs_ref": rel(torch.from_numpy(yo), ref[0].cpu())}
        for nm, a, bb in zip(("gx", "goff", "gw"), go_, ref[1:]):
            r[f"{nm}_oracle_vs_ref"] = rel(torch.from_numpy(a), bb.cpu())
        try:
            mine = run(ours, *cu, k, s, p, d, dg, 0.5)
            for nm, a, bb in zip(("fwd", "gx", "goff", "gw"), mine, ref):
                r[f"{nm}_ours_vs_ref"] = rel(a.cpu(), bb.cpu())
        except Exception as exc:   # keep the golden vectors even if our path is not up yet
            r["ours_error"] = repr(exc)[:300]
        res[name] = r
        print(f"refext_v1 {name}: {json.dumps(r)}", flush=True)
        np.savez_compressed(os.path.join(gold_dir, f"dcn1_ref_cuda_{name}.npz"),
                            x=x.numpy(), offset=off.numpy(), weight=w.numpy(), grad_out=go.numpy(),
                            out=ref[0].cpu().numpy(), grad_x=ref[1].cpu().numpy(), grad_offset=ref[2].cpu().numpy(),
                            grad_weight=ref[3].cpu().numpy(),
                            meta=np.array([N, C, H, W, Cout, dg, *k, *s, *p, *d]), scale=np.float32(0.5))
    return res


def sec_refbench():
    """Time the reference CUDA path (reference dcn ext + cuDNN convs) on EDVR-L cfg 3 and EDVR-M cfg 2."""
    import torch
    from oracle import edvr_ref
    fwd, _ = _ref_fns()
    torch.backends.cudnn.benchmark = True
    res = {"allow_tf32_cudnn": torch.backends.cudnn.allow_tf32, "allow_tf32_matmul": torch.backends.cuda.matmul.allow_tf32}

    def dcn(x, off, mask, w, b, s, p, d, g, dg):
        return fwd(x.contiguous(), off, mask, w, b, s, p, d, g, dg)

    for name, kw, shape in [("cfg2_edvr_m", dict(num_feat=64, num_frame=5, num_reconstruct_block=10), (1, 5, 3, 128, 128)),
                            ("cfg3_edvr_l", dict(num_feat=128, num_frame=7, num_reconstruct_block=40), (1, 7, 3, 180, 320))]:
        sd = {k: v.cuda() for k, v in edvr_ref.make_state_dict(**kw).items()}
        x = torch.rand(*shape, device="cuda")
        for _ in range(3):
            y = edvr_ref.edvr_forward(sd, x, dcn=dcn)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters = 10
        e0.record()
        for _ in range(iters):
            y = edvr_ref.edvr_forward(sd, x, dcn=dcn)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        res[name] = {"ms_per_clip": ms, "fps": 1000.0 / ms, "out_absmax": float(y.abs().max())}
        print(f"refbench {name}: {res[name]}", flush=True)
        # and with torchvision's CUDA deform_conv2d for context
        for _ in range(2):
            y2 = edvr_ref.edvr_forward(sd, x)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            y2 = edvr_ref.edvr_forward(sd, x)
        e1.record()
        torch.cuda.synchronize()
        ms2 = e0.elapsed_time(e1) / iters
        res[name + "_torchvision_dcn"] = {"ms_per_clip": ms2, "fps": 1000.0 / ms2, "vs_refext": rel(y2, y)}
        print(f"refbench {name} (torchvision dcn): {res[name + '_torchvision_dcn']}", flush=True)
    return res


SECTIONS = {"selftest": sec_selftest, "conv": sec_conv, "dcn": sec_dcn, "refext": sec_refext,
            "refext_v1": sec_refext_v1, "refbench": sec_refbench}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--section", default=None)
    ap.add_argument("--only", default=None, help="comma-separated sections for the driver mode")
    a = ap.parse_args()
    if a.section:
        r = SECTIONS[a.section]()
        with open(os.path.join(OUT, f"first_light_{a.section}.json"), "w") as f:
            json.dump(r, f, indent=1)
        return
    names = a.only.split(",") if a.only else list(SECTIONS)
    for name in names:
        t0 = time.time()
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--section", name], timeout=900)
        print(f"== section {name}: exit {p.returncode} in {time.time() - t0:.1f}s", flush=True)


if __name__ == "__main__":
    main()
