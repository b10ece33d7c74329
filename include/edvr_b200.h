/*
 * edvr_b200.h — C ABI of libedvr_b200.so: the B200-native EDVR hot path.
 *
 * Every entry point takes raw DEVICE pointers, explicit sizes and a cudaStream_t (passed as
 * void*), allocates nothing, never synchronises, and returns an int status:
 *   0 ok, -1 invalid shape, -2 unsupported configuration, -3 launch failure,
 *   -4 workspace too small, -5 null pointer, -6 misaligned pointer / stride.
 * (The reference only printf()s launch errors and continues,
 *  /root/reference/basicsr/models/ops/dcn/src/deform_conv_cuda_kernel.cu:794-798.)
 * Calls on different streams may run concurrently; there is no global mutable state.
 *
 * Interface replaced (all paths relative to /root/reference/basicsr/models/):
 *   eb_mdcn_forward / eb_mdcn_backward
 *       == deform_conv_ext.modulated_deform_conv_forward / _backward
 *          (ops/dcn/src/deform_conv_ext.cpp:106-146, bound at ops/dcn/deform_conv.py:141-145,
 *           159-164; implementation ops/dcn/src/deform_conv_cuda.cpp:490-685).
 *          Same tensor layouts (NCHW fp32, offset [N,dg*2*K,Ho,Wo], mask [N,dg*K,Ho,Wo]),
 *          same ownership (caller allocates outputs; grad_weight / grad_bias are accumulated
 *          into, the other grads overwritten), `ones` / `columns` scratch handles dropped in
 *          favour of one caller-owned workspace.
 *   eb_conv2d / eb_dcn_site / eb_dcn_site_pair / eb_* elementwise
 *       == the cuDNN / ATen dispatches behind nn.Conv2d, nn.LeakyReLU, nn.Upsample, nn.*Pool2d,
 *          nn.PixelShuffle, torch.cat in archs/edvr_arch.py:76-117,161-214,250-269,358-420 and
 *          archs/arch_util.py:92-95,243-257, on NHWC fp16 tensors (fp32 accumulation).
 */
#ifndef EDVR_B200_H
#define EDVR_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* activation codes */
#define EB_ACT_NONE 0
#define EB_ACT_RELU 1
#define EB_ACT_LRELU 2      /* negative slope 0.1 (edvr_arch.py:70) */
#define EB_ACT_SIGMOID 4    /* 3 is unassigned: rejected with -2 */
/* output index maps */
#define EB_OUT_SAME 0
#define EB_OUT_PIXSHUF2 1   /* nn.PixelShuffle(2) fused into the store */
#define EB_OUT_STRIDE2 2    /* k3/s2/p1 conv: even-pixel subsample of the stride-1 result */

/* One NHWC fp16 input view of a convolution (channel slice of a wider buffer allowed).
 * Image index used for accumulator image n: (n / div) * mul + (n % div) * keep + add. */
typedef struct {
    const void* ptr;
    int C;            /* channels consumed (multiple of 64) */
    int pix_stride;   /* elements between consecutive pixels (multiple of 8) */
    int ch_off;       /* first channel (multiple of 8) */
    int div, mul, keep, add;
} eb_src_t;

typedef struct {
    const float* bias;        /* [packed Cout] fp32 or NULL */
    int act;
    const void* res16;        /* optional residual, NHWC fp16, added after the activation */
    const float* res32;       /* optional residual, NHWC fp32 */
    int res_pix_stride, res_ch_off;
    void* out16;              /* optional NHWC fp16 output */
    int out16_pix_stride, out16_ch_off;
    float* out32;             /* optional NHWC fp32 output */
    int out32_pix_stride, out32_ch_off;
    float* out_nchw;          /* optional NCHW fp32 output [N][nchw_C][H][W] */
    int nchw_C;
    int out_mode;
    int f32_blocked;          /* res32/out32 use the tile-blocked private layout of eb_f32_blocked_elems() */
    int bf16;                 /* 1: inputs, packed weights and out16 are bf16 instead of fp16 (training step; eb_conv2d_pair,
                                 plain NHWC output only) */
} eb_epilogue_t;

/* ---- library info ------------------------------------------------------------------- */
int eb_version(void);                 /* 100 * major + minor */
const char* eb_last_error(void);      /* thread-local text of the last non-zero status */

/* ---- hardware self-test: D[128,N] = A[128,K] * B[N,K]^T through tcgen05 (fp16 in, fp32 out).
 * variant 0 is the production descriptor convention; other values probe alternatives. */
int eb_selftest_umma(const void* A, const void* B, float* D, int N, int K, int variant, void* stream);
/* Hardware probe (no reference counterpart): cycles per tcgen05.mma for a shape / shared-memory layout / CTA-group
 * choice, `reps` back-to-back MMAs on zeroed operands on every SM; cycles[i] = total cycles seen by CTA i's issuer
 * (0 for non-issuing CTAs of a pair).  layout: 0 no-swizzle planes, 2/4/6 = 128/64/32-byte swizzle. */
int eb_selftest_mma_rate(int cta_group, int M, int N, int layout, int a_lbo, int a_sbo, int b_lbo, int b_sbo,
                         int kstep_bytes, int reps, unsigned long long* cycles, int* n_ctas, void* stream);

/* ---- weight packing (device side; fp32 OIHW -> fp16 MMA-ready stages) ------------------
 * layout [n_tile][chunk][tap][kc=8][BN][8]; packed rows >= cout are zero. */
size_t eb_packed_weight_bytes(int cin, int ktaps, int BN, int n_tiles_n);
int eb_pack_weight(const float* w_oihw, int cout, int cin, int ktaps, int BN, int n_tiles_n, void* wpack, void* stream);

/* ---- dense convolution, NHWC fp16, 3x3 (pad 1) or 1x1, stride 1 (stride 2 via out_mode) ---- */
int eb_conv2d(const eb_src_t* srcs, int nsrc, int N, int H, int W, int ksize, const void* wpack,
              int BN, int n_tiles_n, const eb_epilogue_t* epi, void* stream);
/* same, plus per-CTA cycle counters (device uint64 [148][16]; who waited on which pipeline barrier) */
int eb_conv2d_stats(const eb_src_t* srcs, int nsrc, int N, int H, int W, int ksize, const void* wpack,
                    int BN, int n_tiles_n, const eb_epilogue_t* epi, unsigned long long* stats, void* stream);

/* Same convolution on CTA pairs (tcgen05 cta_group::2), TMA in and out: available when eb_conv2d_pair_supported() is
 * non-zero (Cin % 64 == 0; 1 = each CTA keeps its half of the weights resident in shared memory, 3x3 with
 * Cin * 9 * BN <= 147456, e.g. 128 -> 128; 2 = weights stream with the activation stages: 3x3 256 -> 128, every 1x1).  `wpair` is produced by
 * eb_pack_weight_pair (same size as eb_packed_weight_bytes); sources, epilogue and results as eb_conv2d. */
int eb_conv2d_pair_supported(int cin, int ksize, int BN, int n_tiles_n);
int eb_pack_weight_pair(const float* w, int cout, int cin, int ktaps, int BN, int n_tiles_n, void* wpair, void* stream);
int eb_pack_weight_pair_ex(const float* w, int cout, int cin, int ktaps, int BN, int n_tiles_n, void* wpair, int bf16,
                           void* stream);
/* Weights of the DATA-GRADIENT convolution packed straight from the forward weights w[cout][cin][k][k]: row ci, K index co,
 * tap flipped (training step; k_channels = cout rounded up to a multiple of 64 = channels of the padded grad_out view). */
int eb_pack_weight_pair_dgrad(const float* w, int cout, int cin, int ktaps, int k_channels, int BN, int n_tiles_n, void* wpair,
                              int bf16, void* stream);
int eb_conv2d_pair(const eb_src_t* srcs, int nsrc, int N, int H, int W, int ksize, const void* wpair, int BN,
                   int n_tiles_n, const eb_epilogue_t* epi, void* stream);

/* Tile-blocked fp32 layout of the trunk's residual stream (private to this library: written by eb_tsa_modulate or a
 * conv epilogue, read/updated in place by eb_conv2d epilogues).  Pixels are grouped exactly as the pixel-major conv
 * epilogue owns them (16x16 tiles -> two 16x8 halves -> four 32-pixel quarters -> 32-channel chunks), so that every
 * warp-level float4 access is 512 contiguous bytes.  Returns the number of floats to allocate for [N,H,W,C]. */
size_t eb_f32_blocked_elems(int N, int H, int W, int C);

/* ---- Training step (BASELINE cfg 5): weight gradient of a dense 3x3 (pad 1, stride 1) or 1x1 convolution,
 *   grad_weight[co][ci][ky][kx] += scale * sum_{n,y,x} gy[n,y,x,co] * x[n, y+ky-1, x+kx-1, ci]
 * == the cuDNN wgrad behind autograd of nn.Conv2d in the reference's training loop (basicsr/models/base_model.py:62-69,
 * options/train/EDVR/train_EDVR_L_x4_SR_REDS.yml).  x, gy: NHWC 16-bit views (fp16, or bf16 with bf16 = 1), Cin % 32 == 0;
 * grad_weight fp32 [Cout][Cin][k][k] is ACCUMULATED into (zero it for a plain gradient), deterministically (split-K partial
 * tiles summed in a fixed order); grad_bias, when given, is accumulated while grad_out is transposed.  The data gradient is
 * eb_conv2d_pair on weights packed by eb_pack_weight_pair_dgrad. */
size_t eb_conv_wgrad_workspace(int N, int H, int W, int Cin, int Cout, int ksize);
int eb_conv_wgrad(const void* x, int x_pix_stride, int x_ch_off, const void* gy, int gy_pix_stride, int gy_ch_off, int N,
                  int H, int W, int Cin, int Cout, int ksize, int bf16, float scale, float* grad_weight,
                  float* grad_bias /* optional fp32 [Cout]: += sum of gy over all pixels */, void* workspace,
                  size_t workspace_bytes, void* stream);

/* ---- One DCNv2Pack site (archs/arch_util.py:243-257) for 3x3 / stride 1 / pad 1 / dilation 1 on NHWC fp16 features:
 * the sampled window of x is staged in shared memory by TMA (dcn_site.cuh).  Two ways to supply the offsets:
 *   feat == NULL : `offset` [N][dg*18][H][W] and `mask` [N][dg*9][H][W] (NULL = DCNv1-style, no modulation) in the
 *                  reference's NCHW fp32 channel order (ops/dcn/src/deform_conv_cuda_kernel.cu:600-613), image strides in
 *                  elements; mask_logit = 1 applies the sigmoid of arch_util.py:247 here.
 *   feat != NULL : FUSED - conv_offset (Cin = C -> dg*27, 3x3, pad 1) is computed inside the kernel from the offset
 *                  features `feat` (NHWC fp16 view) with weights from eb_dcn_site_pack_offset_weight; offsets and masks
 *                  never exist in HBM.  offset / mask are ignored.
 * absmean (optional): += sum |offset| over the call, the quantity behind the reference's "offset mean > 50" warning
 * (arch_util.py:249-253), accumulated on the device (no host sync). */
size_t eb_dcn_site_offset_weight_bytes(int C);
int eb_dcn_site_pack_offset_weight(const float* wo /* [dg*27][C][3][3] */, const float* bo /* [dg*27] or NULL */, int C,
                                   int dg, void* wo_pack, float* bo_cols /* [224] */, void* stream);
int eb_dcn_site(const void* x, int x_pix_stride, int x_ch_off, int N, int H, int W, int C, int dg,
                const float* offset, const float* mask, long long off_img_stride, long long mask_img_stride, int mask_logit,
                const void* feat, int f_pix_stride, int f_ch_off, const void* wo_pack, const float* bo_cols,
                const void* wpack, int BN, int n_tiles_n, const eb_epilogue_t* epi, float* absmean, void* stream);

/* ---- CTA-pair form of the fused DCN site (csrc/dcn_pair.cuh): same operation as eb_dcn_site with feat != NULL
 * (DCNv2Pack.forward, arch_util.py:243-257), issued by clusters of two CTAs that split both weight matrices, with the
 * conv_offset GEMM of the next half tile overlapping the gather of the current one.  Needs an even dg with (dg/2)*27 <= 112,
 * C % 64 == 0, C/dg = 8 or a multiple of 16, one output-channel tile (Cout = BN <= 128): eb_dcn_pair_supported() == 1.
 * wpair: the DCN weights packed by eb_pack_weight_pair (n_tiles_n = 1); wo_pack / bo_cols from eb_dcn_pair_pack_offset_weight. */
int eb_dcn_pair_supported(int C, int dg, int BN, int n_tiles_n);
size_t eb_dcn_pair_offset_weight_bytes(int C);
int eb_dcn_pair_pack_offset_weight(const float* wo /* [dg*27][C][3][3] */, const float* bo /* [dg*27] or NULL */, int C,
                                   int dg, void* wo_pack, float* bo_cols /* [224] */, void* stream);
int eb_dcn_site_pair(const void* x, int x_pix_stride, int x_ch_off, int N, int H, int W, int C, int dg,
                     const void* feat, int f_pix_stride, int f_ch_off, const void* wo_pack, const float* bo_cols,
                     const void* wpair, int BN, const eb_epilogue_t* epi, float* absmean, void* stream);
/* development aid: per-role wait-time counters of the pair kernel (all zero unless the library was built with -DDP_PROF) */
int eb_dcn_pair_prof_read(unsigned long long* host32);

/* ---- DCNv2 reference-layout operator (fp32 NCHW in / out) ------------------------------ */
size_t eb_mdcn_forward_workspace(int N, int C, int H, int W, int Cout, int kh, int kw);
int eb_mdcn_forward(const float* x, const float* offset, const float* mask, const float* weight,
                    const float* bias /* NULL = no bias */, float* out, int N, int C, int H, int W,
                    int Cout, int kh, int kw, int stride, int pad, int dil, int groups, int dg,
                    void* workspace, size_t workspace_bytes, void* stream);
/* Half-precision entry (the reference dispatches its kernels on at::Half too: deform_conv_cuda_kernel.cu:781): every tensor
 * fp16 in the reference layouts.  fp16 tensor-core operands (the input as given), fp32 offsets / masks / accumulation, one
 * rounding of the result to fp16.  fp64 tensors have their own entry points (the _f64 functions below). */
size_t eb_mdcn_forward_f16_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, int dg);
int eb_mdcn_forward_f16(const void* x, const void* offset, const void* mask, const void* weight, const void* bias /* or NULL */,
                        void* out, int N, int C, int H, int W, int Cout, int kh, int kw, int stride, int pad, int dil,
                        int groups, int dg, void* workspace, size_t workspace_bytes, void* stream);
size_t eb_mdcn_backward_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, int stride,
                                  int pad, int dil);
int eb_mdcn_backward(const float* x, const float* offset, const float* mask, const float* weight,
                     const float* grad_out, float* grad_x, float* grad_offset, float* grad_mask,
                     float* grad_weight, float* grad_bias /* NULL = no bias */, int N, int C, int H,
                     int W, int Cout, int kh, int kw, int stride, int pad, int dil, int groups, int dg,
                     void* workspace, size_t workspace_bytes, void* stream);

/* ---- DCNv1 (deformable conv without modulation): the other three entry points of the reference extension
 * (deform_conv_ext.cpp:51-104; deform_conv_cuda.cpp:152-488), per-axis stride / pad / dilation like its Python
 * wrapper passes them (deform_conv.py:44-49).  Same NCHW fp32 layouts, offset [N, dg*2*kh*kw, Ho, Wo], no bias.
 * `im2col_step` of the reference is a batching detail with no effect on results and has no equivalent here.
 * Workspace: eb_mdcn_forward_workspace / eb_dcn1_backward_workspace. */
int eb_dcn1_forward(const float* x, const float* offset, const float* weight, float* out, int N, int C, int H, int W,
                    int Cout, int kh, int kw, int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w,
                    int groups, int dg, void* workspace, size_t workspace_bytes, void* stream);
size_t eb_dcn1_backward_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, int stride_h, int stride_w,
                                  int pad_h, int pad_w, int dil_h, int dil_w);
int eb_dcn1_backward_input(const float* x, const float* offset, const float* weight, const float* grad_out, float* grad_x,
                           float* grad_offset, int N, int C, int H, int W, int Cout, int kh, int kw, int stride_h,
                           int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int groups, int dg, void* workspace,
                           size_t workspace_bytes, void* stream);
int eb_dcn1_backward_parameters(const float* x, const float* offset, const float* grad_out, float* grad_weight, float scale,
                                int N, int C, int H, int W, int Cout, int kh, int kw, int stride_h, int stride_w, int pad_h,
                                int pad_w, int dil_h, int dil_w, int groups, int dg, void* workspace, size_t workspace_bytes,
                                void* stream);

/* ---- Double-precision operator (csrc/dcn_f64.cuh): the reference also dispatches on double (deform_conv_cuda_kernel.cu:781,
 * 813,846).  Same layouts, ownership and statuses as the fp32 entries above with double in place of float, and every number
 * stays fp64 (coordinates, bilinear weights, masks, products, accumulators; the GEMMs run on fp64 mma.sync).  Any kh x kw,
 * C, Cout and dg with C % dg == 0 (no C % 64 or Cout limit); groups == 1 (-2 otherwise, as above).  The forwards need no
 * workspace.  The backwards take one of at least the bytes their eb_*_f64_workspace() function returns: the column gradient
 * of a chunk of images for the input side (at least one image; a larger workspace takes more per pass), the split-K
 * partials of grad_weight for the parameter side, the larger of the two for eb_mdcn_backward_f64.  Shapes whose
 * C*kh*kw or Cout exceed 65535 * 64 answer -2.  grad_offset,
 * grad_mask, grad_weight and grad_bias are bit-reproducible; grad_x is an fp64 atomic scatter. */
int eb_mdcn_forward_f64(const double* x, const double* offset, const double* mask, const double* weight,
                        const double* bias /* NULL = no bias */, double* out, int N, int C, int H, int W, int Cout, int kh,
                        int kw, int stride, int pad, int dil, int groups, int dg, void* stream);
size_t eb_mdcn_backward_f64_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, int stride, int pad, int dil);
int eb_mdcn_backward_f64(const double* x, const double* offset, const double* mask, const double* weight,
                         const double* grad_out, double* grad_x, double* grad_offset, double* grad_mask, double* grad_weight,
                         double* grad_bias /* NULL = no bias */, int N, int C, int H, int W, int Cout, int kh, int kw,
                         int stride, int pad, int dil, int groups, int dg, void* workspace, size_t workspace_bytes,
                         void* stream);
int eb_dcn1_forward_f64(const double* x, const double* offset, const double* weight, double* out, int N, int C, int H, int W,
                        int Cout, int kh, int kw, int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w,
                        int groups, int dg, void* stream);
size_t eb_dcn1_backward_input_f64_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, int stride_h, int stride_w,
                                            int pad_h, int pad_w, int dil_h, int dil_w);
size_t eb_dcn1_backward_parameters_f64_workspace(int N, int C, int H, int W, int Cout, int kh, int kw, int stride_h,
                                                 int stride_w, int pad_h, int pad_w, int dil_h, int dil_w);
int eb_dcn1_backward_input_f64(const double* x, const double* offset, const double* weight, const double* grad_out,
                               double* grad_x, double* grad_offset, int N, int C, int H, int W, int Cout, int kh, int kw,
                               int stride_h, int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int groups, int dg,
                               void* workspace, size_t workspace_bytes, void* stream);
int eb_dcn1_backward_parameters_f64(const double* x, const double* offset, const double* grad_out, double* grad_weight,
                                    double scale, int N, int C, int H, int W, int Cout, int kh, int kw, int stride_h,
                                    int stride_w, int pad_h, int pad_w, int dil_h, int dil_w, int groups, int dg,
                                    void* workspace, size_t workspace_bytes, void* stream);

/* ---- layout / elementwise stages of the EDVR graph (all NHWC fp16 unless noted) --------- */
int eb_nchw_f32_to_nhwc_f16(const float* src, void* dst, int N, int C, int H, int W,
                            int dst_pix_stride, int dst_ch_off, void* stream);
int eb_nhwc_f16_to_nchw_f32(const void* src, int src_pix_stride, int src_ch_off, float* dst, int N,
                            int C, int H, int W, void* stream);
/* conv_first: 3x3 pad 1, Cin = 3 (NCHW fp32 frames) -> NHWC fp16, + bias + lrelu */
int eb_conv_first(const float* x_nchw, const float* w_oihw, const float* bias, void* out, int N,
                  int H, int W, int Cout, int out_pix_stride, int act, void* stream);
/* conv_last: 3x3 pad 1, 64 -> 3, + bilinear x4 of the centre LR frame (or + centre frame itself
 * when scale == 1), NCHW fp32 output (edvr_arch.py:413-419) */
int eb_conv_last(const void* x, int x_pix_stride, const float* w_oihw, const float* bias,
                 const float* base_nchw, long long base_img_stride, int scale, float* out_nchw, int N,
                 int H, int W, int Cin, void* stream);
/* out[N, C, H, W] (fp32 NCHW) += bilinear x4 (align_corners = False) of base[N, C, H/4, W/4], or += base when scale == 1:
 * the second half of eb_conv_last for callers that run the 64 -> 3 convolution through eb_conv2d(_pair) with an NCHW store. */
int eb_add_base(const float* base, long long base_img_stride, int scale, float* out, int N, int C, int H, int W, void* stream);
/* bilinear x2, align_corners=False, times `mul` (edvr_arch.py:68-69,109-110), channel-slice I/O */
int eb_upsample2x(const void* src, int src_pix_stride, int src_ch_off, void* dst, int dst_pix_stride,
                  int dst_ch_off, int N, int H, int W, int C, float mul, const void* add,
                  int add_pix_stride, int add_ch_off, void* stream);
/* ---- frame staging either side of the network (SURVEY §8 f2): the arithmetic of read_img_seq after cv2.imread
 * (basicsr/data/data_util.py:28-32 + img2tensor, utils/img_util.py:22-27) and of tensor2img with out_type uint8
 * (utils/img_util.py:62-97), bit-exact.  uint8 images are [N][H][W][C] (OpenCV order, BGR), tensors fp32 [N][C][H][W]. */
int eb_frames_u8_to_f32(const void* hwc_u8, float* chw_f32, int N, int H, int W, int bgr2rgb, void* stream);
int eb_tensor2img_u8(const float* chw_f32, void* hwc_u8, int N, int C /* 1 or 3 */, int H, int W, int rgb2bgr,
                     float lo, float hi, void* stream);
/* MaxPool2d(3,2,1) -> dst[.., 0:C) and AvgPool2d(3,2,1, count_include_pad) -> dst[.., C:2C) */
int eb_pool_max_avg(const void* src, int src_pix_stride, int src_ch_off, void* dst,
                    int dst_pix_stride, int dst_ch_off, int N, int H, int W, int C, void* stream);
/* TSA temporal attention (edvr_arch.py:176-184): prob = sigmoid(sum_c emb[b,t]*emb_ref[b]);
 * dst[b,h,w,t*C+c] = aligned[b*T+t,h,w,c] * prob */
int eb_tsa_temporal(const void* emb, const void* emb_ref, const void* aligned, void* dst, int B, int T,
                    int H, int W, int C, void* stream);
/* TSA output (edvr_arch.py:210-213): out = feat * sigmoid(attn) * 2 + attn_add; fp16 + fp32 copies */
int eb_tsa_modulate(const void* feat, int feat_pix_stride, int feat_ch_off, const void* attn,
                    const void* attn_add, void* out16, float* out32, int N, int H, int W, int C, int f32_blocked,
                    void* stream);
/* dst = a + b (NHWC fp16 views) */
int eb_add(const void* a, int a_pix_stride, int a_ch_off, const void* b, int b_pix_stride,
           int b_ch_off, void* dst, int dst_pix_stride, int dst_ch_off, int npix, int C, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EDVR_B200_H */
