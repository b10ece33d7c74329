"""EDVR forward executor on the B200 kernels (inference path).

Runs the graph of /root/reference/basicsr/models/archs/edvr_arch.py:358-420 (EDVR.forward),
:76-117 (PCDAlignment), :161-214 (TSAFusion), :250-269 (PredeblurModule) and
arch_util.py:92-95,243-257 (ResidualBlockNoBN, DCNv2Pack) from a reference-format state_dict,
but restructured for the hardware:
  * activations NHWC fp16, fp32 accumulation; the 40-block trunk keeps an fp32 residual stream;
  * all T neighbour frames of all B clips go through PCD alignment as ONE batch (the reference
    loops over frames in Python, edvr_arch.py:397-402);
  * torch.cat never materialises: producers write channel slices of a shared buffer, or the conv
    reads two sources (the reference copies up to 59 MB per cat);
  * conv_offset -> (offset, sigmoid(mask)) is one conv whose epilogue emits the packed per-group
    record the DCN kernel consumes; the |offset| mean for the ">50" warning
    (arch_util.py:249-253) is accumulated on the device and read lazily - no host sync per call;
  * feat_fusion and spatial_attn1 (same input, both followed by lrelu) are one 1x1 conv;
  * PixelShuffle, LeakyReLU/ReLU, bias and residual adds live in conv epilogues.
"""
import torch

from . import ops
from .ops import ACT_LRELU, ACT_NONE, ACT_RELU, OUT_PIXSHUF2, OUT_STRIDE2, View


class _Arena:
    """Named persistent device buffers: ONE buffer per name, re-allocated when the requested shape changes, so that
    variable-resolution inference (Vid4, ragged last chunks of forward_video) keeps a single activation set alive instead
    of one multi-GB set per distinct shape."""

    def __init__(self, device):
        self.device = device
        self.bufs = {}

    def _get(self, name, shape, make):
        hit = self.bufs.get(name)
        if hit is None or hit[0] != shape:
            self.bufs.pop(name, None)              # release the old shape before allocating the new one
            hit = self.bufs[name] = (shape, make())
        return hit[1]

    def act(self, name, N, H, W, C, zero=False):
        return View(self._get(name, ("f16", N, H, W, C, zero), lambda: (torch.zeros if zero else torch.empty)(
            N, H, W, C, dtype=torch.float16, device=self.device)))

    def blocked32(self, name, N, H, W, C):
        return self._get(name, ("b32", N, H, W, C), lambda: ops.Blocked32(N, H, W, C, self.device))

    def f32(self, name, *shape):
        return self._get(name, ("f32",) + tuple(shape), lambda: torch.empty(*shape, dtype=torch.float32, device=self.device))


def frame_window_indices(center, n_frames, window, padding="reflection"):
    """Indices of the `window` frames read around `center` in a sequence of n_frames, out-of-range positions folded back by
    `padding` exactly as the reference dataset code does (basicsr/data/data_util.py:35-88; e.g. center 0, window 5:
    replicate 0 0 0 1 2 | reflection 2 1 0 1 2 | reflection_circle 4 3 0 1 2 | circle 3 4 0 1 2)."""
    if window % 2 != 1:
        raise AssertionError("num_frames should be an odd number.")
    if padding not in ("replicate", "reflection", "reflection_circle", "circle"):
        raise AssertionError(f"Wrong padding mode: {padding}.")
    last, half = n_frames - 1, window // 2
    fold_low = {"replicate": lambda i: 0, "reflection": lambda i: -i,
                "reflection_circle": lambda i: center + half - i, "circle": lambda i: window + i}[padding]
    fold_high = {"replicate": lambda i: last, "reflection": lambda i: 2 * last - i,
                 "reflection_circle": lambda i: (center - half) - (i - last), "circle": lambda i: i - window}[padding]
    return [fold_low(i) if i < 0 else fold_high(i) if i > last else i for i in range(center - half, center + half + 1)]


def pack_dcn_site(p, sd, key, dg):
    p[key] = ops.DcnSite(sd[key + ".conv_offset.weight"], sd[key + ".conv_offset.bias"], sd[key + ".weight"],
                         sd.get(key + ".bias"), dg)


def pack_pcd(p, sd, pre, dg):
    """PCDAlignment parameters (edvr_arch.py:21-70) -> MMA-ready packs, keyed by the reference names."""
    for lvl in (3, 2, 1):
        L = f"l{lvl}"
        names = ["offset_conv1." + L, "offset_conv2." + L]
        if lvl < 3:
            names += ["offset_conv3." + L, "feat_conv." + L]
        for n in names:
            p[pre + n] = ops.pack_conv(sd[pre + n + ".weight"], sd.get(pre + n + ".bias"))
        pack_dcn_site(p, sd, pre + "dcn_pack." + L, dg)
    for n in ("cas_offset_conv1", "cas_offset_conv2"):
        p[pre + n] = ops.pack_conv(sd[pre + n + ".weight"], sd.get(pre + n + ".bias"))
    pack_dcn_site(p, sd, pre + "cas_dcnpack", dg)


def pack_tsa(p, sd, pre):
    """TSAFusion parameters (edvr_arch.py:135-159); feat_fusion + spatial_attn1 become one 1x1 conv."""
    for n in ("temporal_attn1", "temporal_attn2", "spatial_attn2", "spatial_attn3", "spatial_attn4",
              "spatial_attn5", "spatial_attn_l1", "spatial_attn_l2", "spatial_attn_l3", "spatial_attn_add1",
              "spatial_attn_add2"):
        p[pre + n] = ops.pack_conv(sd[pre + n + ".weight"], sd.get(pre + n + ".bias"))
    w = torch.cat([sd[pre + "feat_fusion.weight"], sd[pre + "spatial_attn1.weight"]], 0)
    b = torch.cat([sd[pre + "feat_fusion.bias"], sd[pre + "spatial_attn1.bias"]], 0)
    p[pre + "fuse_attn1"] = ops.pack_conv(w, b)


def dcn_site(a, p, key, dg, absmean_slot, x, feat, out, act):
    site = p[key]
    site(x, feat, out, act=act, absmean=absmean_slot, record=site.arena_record(a, feat))


def run_pcd(a, p, pre, dg, absmean, nbr, ref, ref_map, aligned):
    """PCDAlignment.forward (edvr_arch.py:76-117) for a batch of neighbour frames.

    nbr / ref: [L1, L2, L3] Views; the reference image of neighbour n is ref[(n/div)*mul + (n%div)*keep + add]
    with ref_map = (div, mul, keep, add) (None = same index).  absmean: fp32[>=4] device accumulators or None.
    """
    C = nbr[0].C
    N = nbr[0].N
    up_off = up_feat = feat = None
    slot = (lambda i: None) if absmean is None else (lambda i: absmean[i:i + 1])
    for lvl in (3, 2, 1):
        L = f"l{lvl}"
        f, r = nbr[lvl - 1], ref[lvl - 1]
        hh, ww = f.H, f.W
        if lvl == 3:
            o1 = a.act(f"off_a{lvl}", N, hh, ww, C)
            ops.conv2d(p[pre + "offset_conv1." + L], [f, r], out16=o1, act=ACT_LRELU, src_maps=[None, ref_map])
            off = a.act(f"off_b{lvl}", N, hh, ww, C)
            ops.conv2d(p[pre + "offset_conv2." + L], [o1], out16=off, act=ACT_LRELU)
        else:
            ocat = up_off            # [.., 0:C) <- offset_conv1, [.., C:2C) already holds 2*up(offset)
            ops.conv2d(p[pre + "offset_conv1." + L], [f, r], out16=ocat.slice(0, C), act=ACT_LRELU,
                       src_maps=[None, ref_map])
            o2 = a.act(f"off_a{lvl}", N, hh, ww, C)
            ops.conv2d(p[pre + "offset_conv2." + L], [ocat], out16=o2, act=ACT_LRELU)
            off = a.act(f"off_b{lvl}", N, hh, ww, C)
            ops.conv2d(p[pre + "offset_conv3." + L], [o2], out16=off, act=ACT_LRELU)
        if lvl == 3:
            feat = a.act(f"pfeat{lvl}", N, hh, ww, C)
            dcn_site(a, p, pre + "dcn_pack." + L, dg, slot(3 - lvl), f, off, feat, ACT_LRELU)
        else:
            fcat = up_feat           # [.., 0:C) <- dcn output, [.., C:2C) holds up(feat)
            dcn_site(a, p, pre + "dcn_pack." + L, dg, slot(3 - lvl), f, off, fcat.slice(0, C), ACT_NONE)
            feat = a.act(f"pfeat{lvl}", N, hh, ww, C)
            ops.conv2d(p[pre + "feat_conv." + L], [fcat], out16=feat, act=ACT_LRELU if lvl > 1 else ACT_NONE)
        if lvl > 1:
            up_off = a.act(f"ocat{lvl - 1}", N, 2 * hh, 2 * ww, 2 * C)
            up_feat = a.act(f"fcat{lvl - 1}", N, 2 * hh, 2 * ww, 2 * C)
            ops.upsample2x(off, up_off.slice(C, C), mul=2.0)
            ops.upsample2x(feat, up_feat.slice(C, C), mul=1.0)
    h, w = nbr[0].H, nbr[0].W
    c1, c2 = a.act("cas_a", N, h, w, C), a.act("cas_b", N, h, w, C)
    ops.conv2d(p[pre + "cas_offset_conv1"], [feat, ref[0]], out16=c1, act=ACT_LRELU, src_maps=[None, ref_map])
    ops.conv2d(p[pre + "cas_offset_conv2"], [c1], out16=c2, act=ACT_LRELU)
    dcn_site(a, p, pre + "cas_dcnpack", dg, slot(3), feat, c2, aligned, ACT_LRELU)


def run_tsa(a, p, pre, aligned, B, T, center, fused16, trunk32):
    """TSAFusion.forward (edvr_arch.py:161-214); aligned: View [B*T, h, w, C] frame-major per clip."""
    C, h, w = aligned.C, aligned.H, aligned.W
    emb_ref, emb = a.act("emb_ref", B, h, w, C), a.act("emb", B * T, h, w, C)
    ops.conv2d(p[pre + "temporal_attn1"], [aligned], out16=emb_ref, act=ACT_NONE,
               src_maps=[(1, T, 0, center)], N=B)
    ops.conv2d(p[pre + "temporal_attn2"], [aligned], out16=emb, act=ACT_NONE)
    fin = a.act("fus_in", B, h, w, T * C)
    ops.tsa_temporal(emb, emb_ref, aligned, fin, B, T)
    f2 = a.act("fuse2", B, h, w, 2 * C)                   # [0:C) feat, [C:2C) attn
    ops.conv2d(p[pre + "fuse_attn1"], [fin], out16=f2, act=ACT_LRELU)
    h2, w2, h3, w3 = (h + 1) // 2, (w + 1) // 2, ((h + 1) // 2 + 1) // 2, ((w + 1) // 2 + 1) // 2
    p1 = a.act("tsa_p1", B, h2, w2, 2 * C)
    ops.pool_max_avg(f2.slice(C, C), p1)
    a2 = a.act("tsa_a2", B, h2, w2, C)
    ops.conv2d(p[pre + "spatial_attn2"], [p1], out16=a2, act=ACT_LRELU)
    al1 = a.act("tsa_al1", B, h2, w2, C)
    ops.conv2d(p[pre + "spatial_attn_l1"], [a2], out16=al1, act=ACT_LRELU)
    p2 = a.act("tsa_p2", B, h3, w3, 2 * C)
    ops.pool_max_avg(al1, p2)
    al2, al3 = a.act("tsa_al2", B, h3, w3, C), a.act("tsa_al3", B, h3, w3, C)
    ops.conv2d(p[pre + "spatial_attn_l2"], [p2], out16=al2, act=ACT_LRELU)
    ops.conv2d(p[pre + "spatial_attn_l3"], [al2], out16=al3, act=ACT_LRELU)
    al3u = a.act("tsa_al3u", B, 2 * h3, 2 * w3, C)
    ops.upsample2x(al3, al3u)
    assert (2 * h3, 2 * w3) == (h2, w2) and (2 * h2, 2 * w2) == (h, w), "TSA needs h, w multiples of 4"
    a3 = a.act("tsa_a3", B, h2, w2, C)
    ops.conv2d(p[pre + "spatial_attn3"], [a2], out16=a3, act=ACT_LRELU, res16=al3u)
    a4 = a.act("tsa_a4", B, h2, w2, C)
    ops.conv2d(p[pre + "spatial_attn4"], [a3], out16=a4, act=ACT_LRELU)
    a4u = a.act("tsa_a4u", B, h, w, C)
    ops.upsample2x(a4, a4u)
    a5 = a.act("tsa_a5", B, h, w, C)
    ops.conv2d(p[pre + "spatial_attn5"], [a4u], out16=a5, act=ACT_NONE)
    ad1, ad2 = a.act("tsa_ad1", B, h, w, C), a.act("tsa_ad2", B, h, w, C)
    ops.conv2d(p[pre + "spatial_attn_add1"], [a5], out16=ad1, act=ACT_LRELU)
    ops.conv2d(p[pre + "spatial_attn_add2"], [ad1], out16=ad2, act=ACT_NONE)
    ops.tsa_modulate(f2.slice(0, C), a5, ad2, out16=fused16, out32=trunk32)


def unsupported_reasons(sd, C, dg, with_tsa):
    """Why a reference-format state_dict cannot run on the B200 kernels ([] = supported).  There is deliberately no
    PyTorch / cuDNN fallback behind the drop-in modules (north_star): an unsupported configuration is an error."""
    why = []
    if C % 64:
        why.append(f"num_feat={C} must be a multiple of 64 (64-channel K chunks of the implicit GEMMs)")
    if with_tsa and C not in (64, 128, 256):
        why.append(f"num_feat={C}: the TSA correlation kernel covers 64, 128 and 256 channels")
    if dg < 1 or C % dg or not ((C // dg) == 8 or (C // dg) % 16 == 0):
        why.append(f"num_feat/deformable_groups = {C}/{dg} must be 8 or a multiple of 16 (one bilinear sample per 16-byte K atom pair)")
    first = "predeblur.conv_first.weight" if "predeblur.conv_first.weight" in sd else "conv_first.weight"
    if sd[first].shape[1] != 3:
        why.append(f"num_in_ch={sd[first].shape[1]}: conv_first is built for 3 input channels")
    if sd["conv_last.weight"].shape[0] != 3:
        why.append(f"num_out_ch={sd['conv_last.weight'].shape[0]}: the output stage is built for 3 channels")
    return why


class EDVREngine:
    def __init__(self, state_dict, num_frame, center_frame_idx=None, hr_in=False, device="cuda"):
        dev = torch.device(device)
        if dev.type == "cuda" and dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        device = dev
        sd = {k: v.detach().to(device=device, dtype=torch.float32).contiguous() for k, v in state_dict.items()}
        self.device = dev
        self.T = num_frame
        self.center = num_frame // 2 if center_frame_idx is None else center_frame_idx
        self.hr_in = hr_in
        self.C = sd["conv_l2_1.weight"].shape[0]
        self.dg = sd["pcd_align.dcn_pack.l1.conv_offset.weight"].shape[0] // 27
        self.with_predeblur = any(k.startswith("predeblur.") for k in sd)
        self.with_tsa = "fusion.feat_fusion.weight" in sd
        self.n_extract = len({k.split(".")[1] for k in sd if k.startswith("feature_extraction.")})
        self.n_recon = len({k.split(".")[1] for k in sd if k.startswith("reconstruction.")})
        problems = unsupported_reasons(sd, self.C, self.dg, self.with_tsa)
        if problems:
            raise ValueError("edvr_b200 (sm_100a tensor-core path) does not cover this EDVR configuration: " + "; ".join(problems))
        self.arena = _Arena(self.device)
        self.absmean = torch.zeros(16, dtype=torch.float32, device=self.device)   # one slot per DCN site
        self._absmean_counts = None
        self.monitor = ops.OffsetMonitor()      # deferred "Offset abs mean is ..., larger than 50." warning
        self._pack(sd)

    # ------------------------------------------------------------------ weights
    def _pack(self, sd):
        p = {}

        def conv(key):
            p[key] = ops.pack_conv(sd[key + ".weight"], sd.get(key + ".bias"))

        raw = {}
        if self.with_predeblur:
            raw["first"] = (sd["predeblur.conv_first.weight"], sd["predeblur.conv_first.bias"])
            names = ["predeblur.stride_conv_l2", "predeblur.stride_conv_l3", "predeblur.resblock_l3.conv1",
                     "predeblur.resblock_l3.conv2", "predeblur.resblock_l2_1.conv1", "predeblur.resblock_l2_1.conv2",
                     "predeblur.resblock_l2_2.conv1", "predeblur.resblock_l2_2.conv2", "conv_1x1"]
            names += [f"predeblur.resblock_l1.{i}.conv{j}" for i in range(5) for j in (1, 2)]
            if self.hr_in:
                names += ["predeblur.stride_conv_hr1", "predeblur.stride_conv_hr2"]
            for n in names:
                conv(n)
        else:
            raw["first"] = (sd["conv_first.weight"], sd["conv_first.bias"])
        for i in range(self.n_extract):
            conv(f"feature_extraction.{i}.conv1")
            conv(f"feature_extraction.{i}.conv2")
        for n in ("conv_l2_1", "conv_l2_2", "conv_l3_1", "conv_l3_2"):
            conv(n)
        pack_pcd(p, sd, "pcd_align.", self.dg)
        if self.with_tsa:
            pack_tsa(p, sd, "fusion.")
        else:
            conv("fusion")
        for i in range(self.n_recon):
            conv(f"reconstruction.{i}.conv1")
            conv(f"reconstruction.{i}.conv2")
        conv("upconv1")
        conv("upconv2")
        conv("conv_hr")
        raw["last"] = (sd["conv_last.weight"], sd["conv_last.bias"])
        # conv_last on the tensor cores: 3 output channels padded to one 32-wide tile, fp32 NCHW store (+ eb_add_base)
        self.last_tc = ops.pack_conv(sd["conv_last.weight"].float(), sd["conv_last.bias"].float(), cout_packed=32) \
            if sd["conv_last.weight"].shape[1] % 64 == 0 else None
        # conv_first (3 -> C) on the tensor cores: the image goes into channels 0-2 of a zero-filled 64-channel NHWC buffer and
        # the weights are zero-padded to 64 input channels (exact: the extra products are 0); the CUDA-core kernel it replaces
        # was FMA-issue bound at ~3x this time
        wf, bf = raw["first"]
        wpad = torch.zeros(wf.shape[0], 64, 3, 3, dtype=torch.float32, device=wf.device)
        wpad[:, :3] = wf
        self.first_tc = ops.pack_conv(wpad, bf) if wf.shape[0] % 32 == 0 else None
        if self.first_tc is not None:
            self.first_tc.cin_real = 3          # algorithmic FLOPs of conv_first, not of the padded GEMM
        self.p, self.raw = p, raw

    def _first(self, x, out):
        """conv_first + lrelu of an fp32 NCHW image batch into the NHWC fp16 view `out` (edvr_arch.py:371-376,254)."""
        if self.first_tc is None or self.first_tc.wpair is None:
            ops.conv_first(x, *self.raw["first"], out, act=ACT_LRELU)
            return
        N, _, H, W = x.shape
        pad = self.arena.act("first_in", N, H, W, 64, zero=True)
        ops.nchw_to_nhwc(x, out=View(pad.t, 0, 3))
        ops.conv2d(self.first_tc, [pad], out16=out, act=ACT_LRELU)

    # ------------------------------------------------------------------ helpers
    def _resblock16(self, key, x, tmp, out):
        """out = x + conv2(relu(conv1(x))), fp16 residual."""
        ops.conv2d(self.p[key + ".conv1"], [x], out16=tmp, act=ACT_RELU)
        ops.conv2d(self.p[key + ".conv2"], [tmp], out16=out, act=ACT_NONE, res16=x)

    def _submit_offset_check(self):
        self.monitor.submit(self.absmean[:4], self._absmean_counts.tolist(),
                            ["dcn_pack.l3", "dcn_pack.l2", "dcn_pack.l1", "cas_dcnpack"])

    def offset_absmeans(self):
        """Mean |offset| per DCN site of the LAST forward (device sync; the reference warns when > 50)."""
        return None if self._absmean_counts is None else (self.absmean[:4].cpu() / self._absmean_counts)

    # ------------------------------------------------------------------ forward
    def _check_hw(self, hin, win):
        if self.hr_in:
            assert hin % 16 == 0 and win % 16 == 0, "The height and width must be multiple of 16."
        else:
            assert hin % 4 == 0 and win % 4 == 0, "The height and width must be multiple of 4."

    def _features(self, frames):
        """Per-frame pyramid (edvr_arch.py:371-388): fp32 [N,3,hin,win] -> L1/L2/L3 NHWC fp16 views (arena buffers) and (h, w)."""
        a, p, C = self.arena, self.p, self.C
        N, _, hin, win = frames.shape
        if self.with_predeblur:
            l1 = self._predeblur(frames)
            h, w = (hin // 4, win // 4) if self.hr_in else (hin, win)
        else:
            h, w = hin, win
            l1 = a.act("l1a", N, h, w, C)
            self._first(frames, l1)
        tmp, alt = a.act("l1t", N, h, w, C), a.act("l1b", N, h, w, C)
        for i in range(self.n_extract):
            self._resblock16(f"feature_extraction.{i}", l1, tmp, alt)
            l1, alt = alt, l1
        h2, w2, h3, w3 = h // 2, w // 2, h // 4, w // 4
        l2t, l2 = a.act("l2t", N, h2, w2, C), a.act("l2", N, h2, w2, C)
        ops.conv2d(p["conv_l2_1"], [l1], out16=l2t, act=ACT_LRELU, out_mode=OUT_STRIDE2)
        ops.conv2d(p["conv_l2_2"], [l2t], out16=l2, act=ACT_LRELU)
        l3t, l3 = a.act("l3t", N, h3, w3, C), a.act("l3", N, h3, w3, C)
        ops.conv2d(p["conv_l3_1"], [l2], out16=l3t, act=ACT_LRELU, out_mode=OUT_STRIDE2)
        ops.conv2d(p["conv_l3_2"], [l3t], out16=l3, act=ACT_LRELU)
        return l1, l2, l3, h, w

    def _tail(self, l1, l2, l3, B, h, w, base, base_img_stride):
        """PCD alignment, fusion, reconstruction and upsampling for B windows whose B*T frame pyramids are l1/l2/l3
        (edvr_arch.py:390-420).  base: fp32 centre frames, image n at base.data_ptr() + n * base_img_stride elements."""
        a, p, C, T = self.arena, self.p, self.C, self.T
        N = B * T
        h2, w2, h3, w3 = h // 2, w // 2, h // 4, w // 4
        self.absmean.zero_()
        # ---- PCD alignment, all N = B*T neighbour frames at once; reference frame = clip centre
        ref_map = (T, T, 0, self.center)
        self._absmean_counts = torch.tensor([N * h3 * w3, N * h2 * w2, N * h * w, N * h * w],
                                            dtype=torch.float32) * (self.dg * 18)
        aligned = a.act("aligned", N, h, w, C)
        run_pcd(a, p, "pcd_align.", self.dg, self.absmean, [l1, l2, l3], [l1, l2, l3], ref_map, aligned)
        if not torch.cuda.is_current_stream_capturing():
            self._submit_offset_check()

        # ---- fusion
        fused16 = a.act("fused16", B, h, w, C)
        trunk32 = a.blocked32("trunk32", B, h, w, C)      # fp32 residual stream, tile-blocked private layout
        if self.with_tsa:
            run_tsa(a, p, "fusion.", aligned, B, T, self.center, fused16, trunk32)
        else:
            # plain 1x1 over the t*c stack: gather frames into channel-major layout first
            stack = a.act("stack", B, h, w, T * C)
            stack.t.copy_(aligned.t.view(B, T, h, w, C).permute(0, 2, 3, 1, 4).reshape(B, h, w, T * C))
            ops.conv2d(p["fusion"], [stack], out16=fused16, out32=trunk32, act=ACT_NONE)

        # ---- reconstruction trunk: fp32 residual stream + fp16 copy as the next conv input
        x16, y16, t16 = fused16, a.act("trunk_b", B, h, w, C), a.act("trunk_t", B, h, w, C)
        for i in range(self.n_recon):
            ops.conv2d(p[f"reconstruction.{i}.conv1"], [x16], out16=t16, act=ACT_RELU)
            ops.conv2d(p[f"reconstruction.{i}.conv2"], [t16], out16=y16, out32=trunk32, res32=trunk32, act=ACT_NONE)
            x16, y16 = y16, x16

        # ---- upsampler: PixelShuffle + lrelu fused into the conv stores
        u1 = a.act("up1", B, 2 * h, 2 * w, C)
        ops.conv2d(p["upconv1"], [x16], out16=u1, act=ACT_LRELU, out_mode=OUT_PIXSHUF2)
        u2 = a.act("up2", B, 4 * h, 4 * w, 64)
        ops.conv2d(p["upconv2"], [u1], out16=u2, act=ACT_LRELU, out_mode=OUT_PIXSHUF2)
        hr = a.act("hr", B, 4 * h, 4 * w, 64)
        ops.conv2d(p["conv_hr"], [u2], out16=hr, act=ACT_LRELU)
        out = torch.empty(B, 3, 4 * h, 4 * w, dtype=torch.float32, device=self.device)
        if self.last_tc is not None:
            ops.conv2d(self.last_tc, [hr], act=ACT_NONE, out_nchw=out, nchw_C=3)
            ops.add_base(base, base_img_stride, 1 if self.hr_in else 4, out)
        else:
            ops.conv_last(hr, *self.raw["last"], base, base_img_stride, 1 if self.hr_in else 4, out)
        return out

    @torch.no_grad()
    def forward(self, x):
        """x: fp32 [B, T, 3, h, w] on the device -> fp32 [B, 3, 4h, 4w] (or [B,3,h,w] when hr_in)."""
        assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and x.shape[1] == self.T
        assert x.device == self.device, f"input on {x.device}, engine on {self.device}"
        x = x.contiguous()
        B, T, _, hin, win = x.shape
        self._check_hw(hin, win)
        with torch.cuda.device(self.device):       # every launch below uses the current stream of THIS device
            if not torch.cuda.is_current_stream_capturing():
                self.monitor.poll()                # offset warnings of earlier forwards whose read-back has completed
            l1, l2, l3, h, w = self._features(x.view(B * T, 3, hin, win))
            xc = x[:, self.center]          # [B,3,hin,win] view: image stride T*3*hin*win
            return self._tail(l1, l2, l3, B, h, w, xc, T * 3 * hin * win)

    def graphed(self, x):
        """Latency configuration: capture forward() for inputs of x's shape ONCE into a CUDA graph (the ~140 launches of a
        forward, their tensor maps encoded at capture time) and return run(new_x=None) -> output, which replays it.  The
        output tensor and every intermediate live in the graph's private pool; results are bit-identical to forward()."""
        static_x = x.clone()
        with torch.cuda.device(self.device):
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self.forward(static_x)             # allocate arena buffers / load modules outside the capture
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=side):
                    y = self.forward(static_x)
            torch.cuda.current_stream().wait_stream(side)

        def run(new_x=None):
            if new_x is not None:
                static_x.copy_(new_x)
            graph.replay()
            self._submit_offset_check()
            return y
        run.graph, run.output = graph, y
        return run

    @torch.no_grad()
    def forward_video(self, frames, clips_per_step=4, padding="reflection_circle"):
        with torch.cuda.device(self.device):
            return self._forward_video(frames, clips_per_step, padding)

    def _forward_video(self, frames, clips_per_step, padding):
        """Sliding-window inference over one sequence (SURVEY §8 f2): frames fp32 [F, 3, h, w] -> fp32 [F, 3, 4h, 4w], output i
        restored from the window `frame_window_indices(i, F, T, padding)` like the reference's test loop
        (video_base_model.py:44-70 over datasets built with data_util.py:35-88).  The per-frame pyramid (conv_first, feature
        extraction, L2/L3: 24 % of the FLOPs of a clip) is computed ONCE per frame instead of once per window it appears in;
        results are bit-identical to forward() on the explicitly gathered windows."""
        assert frames.is_cuda and frames.dtype == torch.float32 and frames.dim() == 4 and frames.shape[1] == 3
        frames = frames.contiguous()
        F_, _, hin, win = frames.shape
        self._check_hw(hin, win)
        self.monitor.poll()
        T, C, a = self.T, self.C, self.arena
        per_chunk = max(1, clips_per_step * T)
        vid = None
        for s in range(0, F_, per_chunk):
            l1, l2, l3, h, w = self._features(frames[s:s + per_chunk])
            if vid is None:
                vid = [torch.empty(F_, t.H, t.W, C, dtype=torch.float16, device=self.device) for t in (l1, l2, l3)]
            for dst, src in zip(vid, (l1, l2, l3)):
                dst[s:s + src.N].copy_(src.t)
        outs = []
        for c0 in range(0, F_, clips_per_step):
            centers = list(range(c0, min(c0 + clips_per_step, F_)))
            idx = torch.tensor([j for c in centers for j in frame_window_indices(c, F_, T, padding)], device=self.device)
            B = len(centers)
            win_feats = []
            for name, src in zip(("vw1", "vw2", "vw3"), vid):
                dst = a.act(name, B * T, src.shape[1], src.shape[2], C)
                torch.index_select(src, 0, idx, out=dst.t)
                win_feats.append(dst)
            base = frames[centers[0]:centers[-1] + 1]
            outs.append(self._tail(*win_feats, B, h, w, base, 3 * hin * win))
        return torch.cat(outs, 0)

    # ------------------------------------------------------------------ PredeblurModule (edvr_arch.py:250-269)
    def _predeblur(self, x):
        a, p, C = self.arena, self.p, self.C
        N, _, H, W = x.shape
        pre = "predeblur."
        f = a.act("pd_first", N, H, W, C)
        self._first(x, f)
        if self.hr_in:
            f1 = a.act("pd_hr1", N, H // 2, W // 2, C)
            ops.conv2d(p[pre + "stride_conv_hr1"], [f], out16=f1, act=ACT_LRELU, out_mode=OUT_STRIDE2)
            f = a.act("pd_hr2", N, H // 4, W // 4, C)
            ops.conv2d(p[pre + "stride_conv_hr2"], [f1], out16=f, act=ACT_LRELU, out_mode=OUT_STRIDE2)
            H, W = H // 4, W // 4
        l1 = f
        l2 = a.act("pd_l2", N, H // 2, W // 2, C)
        ops.conv2d(p[pre + "stride_conv_l2"], [l1], out16=l2, act=ACT_LRELU, out_mode=OUT_STRIDE2)
        l3 = a.act("pd_l3", N, H // 4, W // 4, C)
        ops.conv2d(p[pre + "stride_conv_l3"], [l2], out16=l3, act=ACT_LRELU, out_mode=OUT_STRIDE2)
        t3, r3 = a.act("pd_t3", N, H // 4, W // 4, C), a.act("pd_r3", N, H // 4, W // 4, C)
        self._resblock16(pre + "resblock_l3", l3, t3, r3)
        t2, r2 = a.act("pd_t2", N, H // 2, W // 2, C), a.act("pd_r2", N, H // 2, W // 2, C)
        self._resblock16(pre + "resblock_l2_1", l2, t2, r2)
        s2 = a.act("pd_s2", N, H // 2, W // 2, C)
        ops.upsample2x(r3, s2, add=r2)                      # resblock_l2_1(l2) + up(l3)
        self._resblock16(pre + "resblock_l2_2", s2, t2, r2)
        t1, b1 = a.act("pd_t1", N, H, W, C), a.act("pd_b1", N, H, W, C)
        cur, other = l1, b1
        for i in range(2):
            self._resblock16(pre + f"resblock_l1.{i}", cur, t1, other)
            cur, other = other, cur
        ops.upsample2x(r2, other, add=cur)                  # l1 + up(l2)
        cur, other = other, cur
        for i in range(2, 5):
            self._resblock16(pre + f"resblock_l1.{i}", cur, t1, other)
            cur, other = other, cur
        out = a.act("l1a", N, H, W, C)
        ops.conv2d(p["conv_1x1"], [cur], out16=out, act=ACT_NONE)
        return out
