"""oracle/make_golden_refext.py — TEST INFRASTRUCTURE ONLY.

Records on a GPU what tests/test_gpu_edvr.py compares the B200 path against: the oracle graph (oracle/edvr_ref.py, the
port of the reference's edvr_arch.py pinned bit for bit by tests/test_oracle.py) with every DCN running the reference's
own CUDA extension, compiled unmodified into oracle/_ref by oracle/build_ref.py.  fp32, TF32 off, cuDNN convolutions.

  l_full_<offset_std>  EDVR-L at full size, 2 clips of 7x3x180x320 -> 3x720x1280
  b1                   EDVR nf 64, 2 clips of 3x3x32x40, multi-pixel offsets

Each output is stored as every `stride`-th element of the flattened tensor (a fixed sample that keeps the file small)
and the max |y| of the whole tensor, in tests/golden/edvr_refext.npz.

Run on a GPU:  python -m oracle.make_golden_refext [OUT_DIR]
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

L_FULL = dict(num_feat=128, num_frame=7, num_extract_block=5, num_reconstruct_block=40)
B1 = dict(num_feat=64, num_frame=3, deformable_groups=8, num_extract_block=1, num_reconstruct_block=2)
# name: (state_dict kwargs, seed, offset_std, input shape, sample stride)
CASES = {f"l_full_{s}": (L_FULL, 9, s, (2, 7, 3, 180, 320), 673) for s in (0.02, 1.0)}
CASES["b1"] = (B1, 21, 1.0, (2, 3, 3, 32, 40), 13)


def ext_dcn(ext):
    """The oracle graph's dcn(...) on a module with the reference's deform_conv_ext signature."""
    def dcn(x, off, mask, w, b, s, p, d, g, dg):
        x = x.contiguous()
        out = x.new_empty(x.shape[0], w.shape[0], x.shape[2], x.shape[3])
        ext.modulated_deform_conv_forward(x, w, b, x.new_empty(0), off, mask, out, x.new_empty(0), 3, 3, s, s, p, p,
                                          d, d, g, dg, True)
        return out
    return dcn


def main():
    sys.path.insert(0, ROOT)
    from oracle import build_ref, edvr_ref
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dcn = ext_dcn(build_ref.load_ref())
    rec = {}
    for name, (kw, seed, offset_std, shape, stride) in CASES.items():
        sd = edvr_ref.make_state_dict(**kw, seed=seed, offset_std=offset_std)
        x = torch.rand(*shape, generator=torch.Generator().manual_seed(seed))
        with torch.no_grad():
            y = edvr_ref.edvr_forward({k: v.cuda() for k, v in sd.items()}, x.cuda(), dcn=dcn)
        rec[name + "_meta"] = np.array([seed, offset_std, stride, *y.shape], np.float64)
        rec[name + "_sample"] = y.flatten()[::stride].cpu().numpy()
        rec[name + "_absmax"] = np.float32(y.abs().max().item())
        print(name, tuple(y.shape), rec[name + "_sample"].size, float(rec[name + "_absmax"]), flush=True)
    os.makedirs(out_dir, exist_ok=True)
    np.savez_compressed(os.path.join(out_dir, "edvr_refext.npz"), **rec)


if __name__ == "__main__":
    main()
