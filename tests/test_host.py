"""CPU tests of the host side: the C-ABI library loads and exports every declared symbol (no compute calls
without a GPU), argument validation that runs before any CUDA call, and the N>1 sharding logic on gloo with world_size 2."""
import ctypes
import json
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_c_abi_exports_match_header():
    from edvr_b200 import build, _lib
    build.build()
    hdr = open(os.path.join(ROOT, "include", "edvr_b200.h")).read()
    declared = set(re.findall(r"\b(eb_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    h = _lib.lib()
    for name in declared:
        assert hasattr(h, name), f"{name} declared in include/edvr_b200.h but not exported"
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    assert h.eb_version() >= 100


def test_host_validation_without_gpu():
    """Argument validation happens before any CUDA call, so it is testable on a CPU-only box."""
    from edvr_b200 import _lib as L
    h = L.lib()
    assert h.eb_mdcn_forward(None, None, None, None, None, None, 1, 64, 8, 8, 64, 3, 3, 1, 1, 1, 1, 8, None, 0, None) == -5
    one = torch.zeros(4)
    p = L.ptr(one)
    assert h.eb_mdcn_forward(p, p, p, p, None, p, 1, 60, 8, 8, 64, 3, 3, 1, 1, 1, 1, 4, None, 0, None) == -2   # C % 64
    assert h.eb_mdcn_forward(p, p, p, p, None, p, 1, 64, 8, 8, 64, 3, 3, 1, 1, 1, 2, 8, None, 0, None) == -2   # groups
    assert h.eb_mdcn_forward(p, p, p, p, None, p, 1, 64, 8, 8, 64, 3, 3, 0, 1, 1, 1, 8, None, 0, None) == -1   # stride 0
    assert h.eb_mdcn_forward(p, p, p, p, None, p, 1, 64, 8, 8, 64, 3, 3, 1, 1, 1, 1, 8, None, 0, None) == -4   # workspace
    assert b"workspace" in h.eb_last_error()
    assert h.eb_mdcn_forward_workspace(1, 64, 8, 8, 64, 3, 3) >= 8 * 8 * 64 * 2
    assert h.eb_packed_weight_bytes(128, 9, 128, 1) == 128 * 128 * 9 * 2
    # activation code 3 is unassigned: the epilogue check rejects it before the kernel choice touches the device
    src = (L.Src * 1)(L.Src(p.value, 64, 64, 0, 1, 1, 0, 0))
    e = L.Epilogue(act=3, out16=p.value, out16_pix_stride=64)
    assert h.eb_conv2d(src, 1, 1, 8, 8, 3, p, 128, 1, ctypes.byref(e), None) == -2
    assert h.eb_conv2d_pair(src, 1, 1, 8, 8, 3, p, 128, 1, ctypes.byref(e), None) == -2
    assert b"act 3" in h.eb_last_error()


def test_dcn_site_rejects_unknown_mode(monkeypatch):
    """A mode outside pair / fused / split is an error, raised before any packing or CUDA call (CPU tensors here)."""
    from edvr_b200.ops import DcnSite
    wo, w = torch.zeros(8 * 27, 64, 3, 3), torch.zeros(64, 64, 3, 3)
    with pytest.raises(ValueError, match="'legacy'"):
        DcnSite(wo, None, w, None, 8, mode="legacy")
    monkeypatch.setenv("EDVR_B200_DCN_SITE", "legacy")
    with pytest.raises(ValueError, match="'legacy'"):
        DcnSite(wo, None, w, None, 8)


def test_missing_library_fails_loudly(monkeypatch):
    from edvr_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libedvr_b200.so")
    with pytest.raises(RuntimeError, match="no fallback"):
        _lib.lib()


def test_cpu_tensors_raise_like_reference():
    from edvr_b200.dcn import modulated_deform_conv
    with pytest.raises(NotImplementedError):
        modulated_deform_conv(torch.zeros(1, 64, 4, 4), torch.zeros(1, 144, 4, 4), torch.zeros(1, 72, 4, 4),
                              torch.zeros(64, 64, 3, 3), None, 1, 1, 1, 1, 8)


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from edvr_b200 import shard
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    mine = shard.clip_shard(7, rank, world)
    mx = shard.reduce_max(10.0 + rank)
    sm = shard.reduce_sum(len(mine))
    q.put((rank, mine, mx, sm))
    dist.destroy_process_group()


def test_sharding_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 500
    ps = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = sorted(q.get(timeout=120) for _ in ps)
    for p in ps:
        p.join(60)
    assert res[0][1] == [0, 2, 4, 6] and res[1][1] == [1, 3, 5]
    assert all(r[2] == 11.0 for r in res) and all(r[3] == 7.0 for r in res)   # max over ranks, every clip once


def _ref_host(golden_dir):
    with open(os.path.join(golden_dir, "ref_host.json")) as f:
        return json.load(f)


def test_reference_tree_imports_unchanged_with_b1_shim(golden_dir):
    """Registering edvr_b200.deform_conv_ext as the compiled module lets the reference tree import and construct EDVR
    with its own ModulatedDeformConvPack (SURVEY App. B).  Pinned by tests/golden/ref_host.json (oracle/make_golden_live.py,
    recorded from the reference with the shim registered): every deform_conv_ext call of the reference's dcn layer binds
    to the shim's function of that name with the same positional argument count, and the drop-in EDVR has the state_dict
    keys and shapes of the reference EDVR built on the shim."""
    import inspect
    import edvr_b200.deform_conv_ext as ext
    from edvr_b200.edvr import EDVR
    ref = _ref_host(golden_dir)
    assert len(ref["ext_calls"]) == 5
    for name, nargs in ref["ext_calls"].items():
        inspect.signature(getattr(ext, name)).bind(*range(nargs))
    want = ref["shim_edvr"]["state_dict"]
    assert len(want) > 50
    got = {k: list(v.shape) for k, v in EDVR(**ref["shim_edvr"]["kwargs"]).state_dict().items()}
    assert got == want


def test_checkpoint_wire_format_roundtrip(tmp_path):
    """SURVEY §8 f4: the reference's checkpoint format ({'params': state_dict}, optional 'module.' prefixes,
    base_model.py:171-262) loads into the drop-in EDVR with strict=True and is written back in the same format."""
    from edvr_b200.edvr import EDVR, load_network, save_network
    from oracle import edvr_ref
    kw = dict(num_feat=64, num_frame=3, deformable_groups=8, num_extract_block=1, num_reconstruct_block=2)
    sd = edvr_ref.make_state_dict(**kw, seed=3)
    path = tmp_path / "EDVR_ckpt.pth"
    torch.save({"params": {"module." + k: v for k, v in sd.items()}}, path)          # as saved from a DataParallel wrapper
    net = load_network(EDVR(center_frame_idx=None, **kw), str(path), strict=True)
    got = net.state_dict()
    assert set(got) == set(sd) and all(torch.equal(got[k], sd[k]) for k in sd)
    out = tmp_path / "resaved.pth"
    save_network(net, str(out))
    back = torch.load(out)
    assert set(back) == {"params"} and all(torch.equal(back["params"][k], sd[k]) for k in sd)
    # strict=False skips tensors whose size differs (base_model.py:229-236) instead of raising
    bad = dict(sd)
    bad["conv_first.weight"] = torch.zeros(64, 3, 5, 5)
    torch.save({"params": bad}, path)
    load_network(EDVR(center_frame_idx=None, **kw), str(path), strict=False)
    with pytest.raises(RuntimeError):
        load_network(EDVR(center_frame_idx=None, **kw), str(path), strict=True)


def test_frame_window_indices_follow_reference_padding_modes(golden_dir):
    """The four padding modes of the reference's sequence datasets (examples of data_util.py:46-53) and every
    (mode, length, window, centre) against its generate_frame_indices, recorded in tests/golden/ref_host.json."""
    from edvr_b200.engine import frame_window_indices as f
    assert f(0, 100, 5, "replicate") == [0, 0, 0, 1, 2]
    assert f(0, 100, 5, "reflection") == [2, 1, 0, 1, 2]
    assert f(0, 100, 5, "reflection_circle") == [4, 3, 0, 1, 2]
    assert f(0, 100, 5, "circle") == [3, 4, 0, 1, 2]
    assert f(99, 100, 5, "reflection") == [97, 98, 99, 98, 97]
    assert f(50, 100, 7, "reflection") == list(range(47, 54))
    with pytest.raises(AssertionError):
        f(0, 10, 4)
    with pytest.raises(AssertionError):
        f(0, 10, 5, "zeros")
    ref = _ref_host(golden_dir)["frame_windows"]
    assert (ref["paddings"], ref["lengths"], ref["windows"]) == (["replicate", "reflection", "reflection_circle", "circle"],
                                                                 [7, 10, 33], [3, 5, 7])
    for pad in ref["paddings"]:
        for n in ref["lengths"]:
            for t in ref["windows"]:
                want = ref["indices"][pad][str(n)][str(t)]
                assert len(want) == n and all(f(c, n, t, pad) == want[c] for c in range(n)), (pad, n, t)


def test_official_key_map_matches_reference_conversion_script(golden_dir):
    """edvr_b200.edvr.official_key vs the key map of the reference's own convert_edvr() (scripts/model_conversion), run
    unmodified with torch.load / torch.save intercepted - the 'official' checkpoint answers every lookup with the
    requested key name, so the saved dict IS the map - and recorded in tests/golden/ref_host.json."""
    from edvr_b200.edvr import official_key
    from oracle import edvr_ref
    maps = _ref_host(golden_dir)["official_key_maps"]
    assert len(maps) == 3
    for entry in maps:
        keys = list(edvr_ref.make_state_dict(**entry["kwargs"]))
        saved = entry["map"]
        assert set(saved) == set(keys)
        for k in keys:
            assert official_key(k) == saved[k], (k, official_key(k), saved[k])


def test_group_slices_compose_a_grouped_dcn_from_single_group_calls():
    """Host logic of the weight-group composition (edvr_b200.ops.group_slices, used by the B1 / B2 boundary for groups > 1;
    deform_conv_cuda.cpp:536-568): running the ORACLE once per slice with groups = 1 and concatenating must equal the oracle's
    own grouped forward, for deformable groups that are a multiple of the weight groups and for shared deformable groups."""
    import numpy as np
    import torch
    from edvr_b200.ops import group_slices
    from oracle import dcn_oracle
    g = torch.Generator().manual_seed(4)
    N, C, H, W, Cout = 1, 16, 6, 7, 8
    for groups, dg in ((2, 2), (2, 4), (4, 2), (2, 1)):
        x = torch.randn(N, C, H, W, generator=g).numpy()
        off = (torch.randn(N, dg * 18, H, W, generator=g) * 2).numpy()
        mask = torch.rand(N, dg * 9, H, W, generator=g).numpy()
        w = torch.randn(Cout, C // groups, 3, 3, generator=g).numpy()
        b = torch.randn(Cout, generator=g).numpy()
        want = dcn_oracle.forward(x, off, mask, w, b, 1, 1, 1, groups, dg)
        parts = []
        for gi in range(groups):
            cs, os_, fs, ms, dgg = group_slices(C, Cout, 9, groups, dg, gi)
            parts.append(dcn_oracle.forward(np.ascontiguousarray(x[:, cs]), np.ascontiguousarray(off[:, fs]),
                                            np.ascontiguousarray(mask[:, ms]), np.ascontiguousarray(w[os_]),
                                            np.ascontiguousarray(b[os_]), 1, 1, 1, 1, dgg))
        got = np.concatenate(parts, 1)
        assert np.abs(got - want).max() < 1e-5 * np.abs(want).max(), (groups, dg)
    with pytest.raises(RuntimeError, match="one must divide the other"):
        group_slices(24, 24, 9, 2, 3, 0)


def test_frame_staging_has_no_cpu_fallback():
    import torch
    from edvr_b200 import frames_to_tensor, tensor2img, tensor_to_bytes
    with pytest.raises(NotImplementedError):
        tensor2img(torch.zeros(3, 4, 4))
    with pytest.raises(NotImplementedError):
        frames_to_tensor(torch.zeros(1, 4, 4, 3, dtype=torch.uint8))
    with pytest.raises(NotImplementedError):
        tensor_to_bytes(torch.zeros(1, 3, 4, 4))
    with pytest.raises(TypeError):
        tensor2img(3.0)
