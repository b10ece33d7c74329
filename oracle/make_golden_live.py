"""oracle/make_golden_live.py — TEST INFRASTRUCTURE ONLY.

Records, from an unmodified checkout of the reference (BasicSR), what the host-side tests compare against, so that the
tests run without that checkout:

  tests/golden/ref_host.json   positional-argument count of every deform_conv_ext call in the reference's dcn Python
                               layer; state_dict key -> shape of the reference EDVR built with edvr_b200.deform_conv_ext
                               registered as its compiled module; generate_frame_indices for every (padding, sequence
                               length, window, centre) the test checks; the key map of the reference's convert_edvr();
                               the state_dict keys of the reference EDVR in the live port comparison
  tests/golden/ref_live.npz    the reference EDVR graph's output on one seeded input (port comparison) and the
                               reference's img2tensor / tensor2img on seeded frames and outputs

Run:  python -m oracle.make_golden_live REFERENCE_DIR
"""
import ast
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, "tests", "golden")

SHIM_EDVR = dict(num_feat=64, num_frame=3, num_reconstruct_block=1, center_frame_idx=None)
PORT_EDVR = dict(num_feat=16, num_frame=3, deformable_groups=2, num_extract_block=1, num_reconstruct_block=1, with_tsa=True)
PORT_SEED = 4
FRAME_WINDOWS = dict(paddings=("replicate", "reflection", "reflection_circle", "circle"), lengths=(7, 10, 33),
                     windows=(3, 5, 7))
KEY_MAP_CONFIGS = (dict(num_feat=64, num_frame=3, num_extract_block=1, num_reconstruct_block=2),
                   dict(num_feat=64, num_frame=3, num_extract_block=1, num_reconstruct_block=1, with_tsa=False),
                   dict(num_feat=64, num_frame=3, num_extract_block=1, num_reconstruct_block=1, with_predeblur=True,
                        hr_in=True))


def ext_calls(ref):
    """{function: positional argument count} of every `deform_conv_ext.<function>(...)` in the reference's dcn layer."""
    tree = ast.parse(open(os.path.join(ref, "basicsr", "models", "ops", "dcn", "deform_conv.py")).read())
    calls = {}
    for node in ast.walk(tree):
        f = getattr(node, "func", None)
        if isinstance(node, ast.Call) and isinstance(f, ast.Attribute) and getattr(f.value, "id", None) == "deform_conv_ext":
            assert not node.keywords and calls.get(f.attr, len(node.args)) == len(node.args), f.attr
            calls[f.attr] = len(node.args)
    return calls


def shim_edvr_state_dict(ref):
    """The reference's EDVR constructed with edvr_b200.deform_conv_ext as its compiled dcn module."""
    import edvr_b200.deform_conv_ext as ext
    sys.modules["basicsr.models.ops.dcn.deform_conv_ext"] = ext
    from basicsr.models.archs import arch_util, edvr_arch
    from basicsr.models.ops.dcn.deform_conv import ModulatedDeformConvPack
    assert arch_util.DCNv2Pack.__mro__[1] is ModulatedDeformConvPack
    net = edvr_arch.EDVR(**SHIM_EDVR)
    return {k: list(v.shape) for k, v in net.state_dict().items()}


def frame_indices(ref):
    src = open(os.path.join(ref, "basicsr", "data", "data_util.py")).read()
    ns = {}
    exec(src[src.index("def generate_frame_indices"):src.index("def paired_paths_from_lmdb")], ns)
    gen = ns["generate_frame_indices"]
    return {pad: {str(n): {str(t): [gen(c, n, t, pad) for c in range(n)] for t in FRAME_WINDOWS["windows"]}
                  for n in FRAME_WINDOWS["lengths"]} for pad in FRAME_WINDOWS["paddings"]}


def official_key_maps(ref):
    """convert_edvr() run unmodified with torch.load / torch.save intercepted: the 'official' checkpoint answers every
    lookup with the requested key name, so the saved dict is the key map."""
    import importlib.util
    from oracle import edvr_ref
    spec = importlib.util.spec_from_file_location("ref_convert_models",
                                                  os.path.join(ref, "scripts", "model_conversion", "convert_models.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)

    class Echo(dict):
        def __missing__(self, k):
            return k

    maps = []
    load, save = mod.torch.load, mod.torch.save
    try:
        for kw in KEY_MAP_CONFIGS:
            keys = list(edvr_ref.make_state_dict(**kw))
            loads = iter([Echo(), {k: None for k in keys}])
            saved = {}
            mod.torch.load = lambda *a, **k: next(loads)
            mod.torch.save = lambda obj, path: saved.update(obj)
            mod.convert_edvr()
            maps.append({"kwargs": kw, "map": saved})
    finally:
        mod.torch.load, mod.torch.save = load, save
    return maps


def main():
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "basicsr")):
        sys.exit(__doc__)
    ref = os.path.abspath(sys.argv[1])
    sys.dont_write_bytecode = True
    sys.path[:0] = [ref, ROOT]
    from oracle import make_golden_img
    from oracle.make_golden import RECORDING_THREADS, reference_edvr
    torch.set_num_threads(RECORDING_THREADS)

    host = {"ext_calls": ext_calls(ref), "shim_edvr": {"kwargs": SHIM_EDVR, "state_dict": shim_edvr_state_dict(ref)},
            "frame_windows": dict(FRAME_WINDOWS, indices=frame_indices(ref)), "official_key_maps": official_key_maps(ref)}

    net, _ = reference_edvr(PORT_EDVR, seed=PORT_SEED)          # DCN through torchvision's CPU deform_conv2d
    x = torch.rand(1, 3, 3, 8, 12, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        y = net(x)
    host["port_edvr"] = {"kwargs": PORT_EDVR, "seed": PORT_SEED, "state_dict_keys": sorted(net.state_dict())}

    img2tensor, tensor2img = make_golden_img.reference_functions()
    rng = np.random.default_rng(3)
    frames = rng.integers(0, 256, size=(2, 9, 11, 3), dtype=np.uint8)
    img_x = torch.stack(img2tensor([f.astype(np.float32) / 255. for f in frames], bgr2rgb=True, float32=True), 0).numpy()
    img_out = rng.normal(0.5, 0.6, size=(1, 3, 13, 7)).astype(np.float32)

    with open(os.path.join(OUT, "ref_host.json"), "w") as f:
        json.dump(host, f, indent=None, separators=(",", ":"), sort_keys=True)
        f.write("\n")
    np.savez_compressed(os.path.join(OUT, "ref_live.npz"), edvr_x=x.numpy(), edvr_y=y.numpy(),
                        img_frames=frames, img_x=img_x, img_out=img_out,
                        img_y=tensor2img(torch.from_numpy(img_out)), img_y00=tensor2img(torch.from_numpy(img_out[0, 0])))
    print("wrote ref_host.json, ref_live.npz:", {k: len(v) for k, v in host.items() if isinstance(v, (dict, list))})


if __name__ == "__main__":
    main()
