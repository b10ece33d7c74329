"""oracle/make_golden.py — TEST INFRASTRUCTURE ONLY.

Generates tests/golden/edvr_ref_import_*.npz by importing the UNMODIFIED reference Python graph from
/root/reference (read-only) in the build container, with the dcn B1 extension stubbed and the B2 op
bound to torchvision's CPU deform_conv2d (SURVEY App. B).  Run:  python -m oracle.make_golden
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")
# intra-op threads of every CPU graph recording: the CPU convolutions split their reductions by thread count, so a
# bit-exact comparison with a recording runs with the same count (tests/test_oracle.py)
RECORDING_THREADS = 8


def reference_edvr(kwargs, seed):
    """Build basicsr.models.archs.edvr_arch.EDVR(**kwargs) with synthetic weights; returns (net, state_dict)."""
    if "/root/reference" not in sys.path:
        sys.path.insert(0, "/root/reference")
    sys.dont_write_bytecode = True
    name = "basicsr.models.ops.dcn.deform_conv_ext"
    if name not in sys.modules:
        stub = types.ModuleType("deform_conv_ext")
        for fn in ("deform_conv_forward", "deform_conv_backward_input", "deform_conv_backward_parameters",
                   "modulated_deform_conv_forward", "modulated_deform_conv_backward"):
            setattr(stub, fn, None)
        sys.modules[name] = stub
    from basicsr.models.archs import arch_util, edvr_arch
    from oracle import edvr_ref
    arch_util.modulated_deform_conv = edvr_ref.dcn_torchvision
    net = edvr_arch.EDVR(center_frame_idx=None, **kwargs).eval()
    sd = edvr_ref.make_state_dict(**kwargs, seed=seed)
    net.load_state_dict(sd, strict=True)
    return net, sd


CASES = {
    "tsa": (dict(num_feat=16, num_frame=3, deformable_groups=2, num_extract_block=2, num_reconstruct_block=2,
                 with_tsa=True), (1, 3, 3, 16, 24)),
    "notsa": (dict(num_feat=16, num_frame=5, deformable_groups=4, num_extract_block=1, num_reconstruct_block=1,
                   with_tsa=False), (2, 5, 3, 8, 12)),
    "predeblur_hr": (dict(num_feat=16, num_frame=3, deformable_groups=2, num_extract_block=1,
                          num_reconstruct_block=1, with_tsa=True, with_predeblur=True, hr_in=True), (1, 3, 3, 32, 48)),
    # the smallest configuration the tensor-core path supports (num_feat multiple of 64)
    "nf64": (dict(num_feat=64, num_frame=3, deformable_groups=8, num_extract_block=1, num_reconstruct_block=2,
                  with_tsa=True), (1, 3, 3, 16, 16)),
}


def main():
    torch.set_num_threads(RECORDING_THREADS)
    os.makedirs(OUT, exist_ok=True)
    for name, (kw, shape) in CASES.items():
        net, _ = reference_edvr(kw, seed=11)
        x = torch.rand(*shape, generator=torch.Generator().manual_seed(5))
        with torch.no_grad():
            y = net(x)
        np.savez_compressed(os.path.join(OUT, f"edvr_ref_import_{name}.npz"), x=x.numpy(), y=y.numpy(),
                            kwargs=np.array(kw, dtype=object), seed=11)
        print(name, tuple(y.shape), float(y.abs().max()))


if __name__ == "__main__":
    main()
