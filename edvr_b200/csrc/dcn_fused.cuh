// dcn_fused.cuh — DCNv2 (modulated deformable convolution) forward, one fused kernel.
//
// Replaces modulated_deform_conv_cuda_forward + modulated_deformable_im2col_gpu_kernel + the
// per-sample addmm_ + the bias pass
// (/root/reference/basicsr/models/ops/dcn/src/deform_conv_cuda.cpp:490-569,
//  deform_conv_cuda_kernel.cu:467-497,570-633): the im2col "columns" matrix never exists in
// HBM.  For each tile of 16x8 output pixels, the gather warps bilinear-sample the NHWC fp16
// input (16 B = 8 channels per corner load), apply the modulation mask and write the result
// straight into the shared-memory A operand (no-swizzle K-major planes, common.cuh); one
// thread issues tcgen05.mma against the pre-packed weights (B operand, bulk async copies);
// the fp32 accumulator lives in TMEM and is drained by four epilogue warps (bias, NCHW fp32
// store).  Offsets and masks arrive fp32 NCHW in the reference layout.  K is walked chunk-major: stage = (64-channel chunk, tap), so the nine
// taps of a chunk re-read the same ~23 KB slab of x and hit L1.
// Gather mapping (L1TEX wavefronts and issue slots are the limiters of this kernel, profiles/r01_*): four lanes
// read the 128 contiguous bytes (64 channels) of ONE sampled pixel per corner, each lane 32 bytes = one
// deformable group when C/dg = 16, so the sampling geometry is computed once per 16 channels; offsets of the next
// stage are prefetched while the current one is gathered.
//
// Sampling semantics (bit-for-bit the reference's decisions, fp32 coordinate math):
//   h_im = ho*stride - pad + i*dil + dh;  sample iff h_im > -1 && w_im > -1 && h_im < H && w_im < W
//   corners outside [0,H-1]x[0,W-1] contribute 0; floor() picks the low corner.
#pragma once
#include "common.cuh"
#include "epilogue.cuh"

namespace eb {

constexpr int DC_STAGES = 4;             // 4 x 32 KB: leaves ~90 KB of the SM's L1 for the gather
constexpr int DC_A_LBO = 128 * 16 + 16;  // plane pitch (+16 B: the 8 kc-lanes of a pixel hit 8 different bank groups)
constexpr int DC_A_BYTES = 8 * DC_A_LBO; // 8 planes x 128 rows x 16 B (+ pad)
constexpr int DC_B_BYTES = 128 * 128;    // BN(<=128) rows x 64 ch x 2 B
constexpr int DC_NPX = 1;                // output pixels per gather thread and stage.  1 -> 16 gather warps (4 per scheduler):
                                         // the gather is latency/issue bound, twice the warps hide more than 2-pixel ILP did
constexpr int DC_GATHER_THREADS = 512 / DC_NPX;
constexpr int DC_THREADS = 192 + DC_GATHER_THREADS + 32;   // warps 0 B-producer, 1 MMA, 2-5 epilogue, 6.. gather, last: forwarder
constexpr int DC_MAX_COUT = 512;
constexpr int DC_SMEM_BYTES = DC_STAGES * (DC_A_BYTES + DC_B_BYTES) + DC_MAX_COUT * 4 + 256;
constexpr int DC_TILE_H = 16, DC_TILE_W = 8;

struct DcnParams {
    const __half* x;          // NHWC fp16 [N][H][W][C] view
    int x_pix_stride, x_ch_off;
    int x_wide;               // 1: every (pixel, 16-channel group) of the view is 32-byte aligned -> one LDG.256 per corner
    int N, H, W, C;
    int Ho, Wo;
    int kh, kw, stride, pad, dil;   // along H
    int stride_w, pad_w, dil_w;     // along W (DCNv1 passes independent pairs; v2 passes equal values)
    int dg, cpg;              // deformable groups, channels per group (multiple of 8)
    const float* offset;      // [N][dg*2*K][Ho][Wo]   (reference layout)
    const float* mask;        // [N][dg*K][Ho][Wo]; NULL = no modulation (DCNv1)
    const __half* wpack;      // [n_tile][chunk][tap][kc=8][BN][8] fp16
    int BN, n_tiles_n;
    EpiParams epi;            // epi.H/W == Ho/Wo
};

struct DcnCorner {
    float w[4];
    int off[4];           // element offset of each corner from the image base (channel 0 of the view); -1: contributes 0
};

// corners that contribute nothing are read from here: unconditional loads, no zero-initialised registers, no NaN hazard
__device__ __align__(32) const uint32_t dcn_zero32[8] = {0, 0, 0, 0, 0, 0, 0, 0};

struct DcnOff { float dh, dw, mk; };

__device__ __forceinline__ void dcn_blend8(float (&acc)[8], uint4 u, float w) {
    const float2 a = unpack_h2(u.x), b = unpack_h2(u.y), c = unpack_h2(u.z), d = unpack_h2(u.w);
    acc[0] = fmaf(w, a.x, acc[0]); acc[1] = fmaf(w, a.y, acc[1]);
    acc[2] = fmaf(w, b.x, acc[2]); acc[3] = fmaf(w, b.y, acc[3]);
    acc[4] = fmaf(w, c.x, acc[4]); acc[5] = fmaf(w, c.y, acc[5]);
    acc[6] = fmaf(w, d.x, acc[6]); acc[7] = fmaf(w, d.y, acc[7]);
}

__global__ void __launch_bounds__(DC_THREADS, 1) dcn_fused_kernel(const DcnParams P) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* a_smem = smem;
    uint8_t* b_smem = smem + DC_STAGES * DC_A_BYTES;
    float* bias_s = reinterpret_cast<float*>(b_smem + DC_STAGES * DC_B_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(bias_s + DC_MAX_COUT);
    uint64_t* full = bars;                       // [S]  forwarder arrival + 1 expect_tx (weights)
    uint64_t* empty = bars + DC_STAGES;          // [S]
    uint64_t* gathered = bars + 2 * DC_STAGES;   // [S]  one arrival per gather warp
    uint64_t* acc_full = bars + 3 * DC_STAGES;   // [2]
    uint64_t* acc_empty = acc_full + 2;          // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_x = (P.Wo + DC_TILE_W - 1) / DC_TILE_W;
    const int tiles_y = (P.Ho + DC_TILE_H - 1) / DC_TILE_H;
    const int total_tiles = P.N * tiles_y * tiles_x * P.n_tiles_n;
    const int nchunks = P.C / 64;
    const int K = P.kh * P.kw;
    const int nstages = K * nchunks;
    const uint32_t b_bytes = static_cast<uint32_t>(P.BN) * 128u;

    const int cout_packed = P.BN * P.n_tiles_n;
    const bool has_bias = P.epi.bias != nullptr;
    if (has_bias)
        for (int i = threadIdx.x; i < cout_packed; i += blockDim.x) bias_s[i] = P.epi.bias[i];
    if (threadIdx.x == 0) {
        for (int i = 0; i < DC_STAGES; ++i) { mbar_init(&full[i], 2); mbar_init(&empty[i], 1); mbar_init(&gathered[i], DC_GATHER_THREADS / 32); }
        for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 4); }
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, 256);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= B producer
        if (lane == 0) {
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int nt = tile % P.n_tiles_n;
                const uint8_t* w = reinterpret_cast<const uint8_t*>(P.wpack) +
                                   static_cast<size_t>(nt) * nstages * b_bytes;
                for (int st = 0; st < nstages; ++st, ++it) {
                    const uint32_t s = it % DC_STAGES, ph = (it / DC_STAGES) & 1u;
                    mbar_wait(&empty[s], ph ^ 1u);
                    mbar_arrive_expect_tx(&full[s], b_bytes);
                    bulk_g2s(b_smem + s * DC_B_BYTES, w + static_cast<size_t>(st) * b_bytes, b_bytes, &full[s]);
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_f16(128, P.BN);
            const uint32_t lbo_b = static_cast<uint32_t>(P.BN) * 16u;
            uint32_t it = 0, acc_it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++acc_it) {
                const uint32_t ab = acc_it & 1u;
                mbar_wait(&acc_empty[ab], ((acc_it >> 1) & 1u) ^ 1u);
                tc_fence_after_sync();
                const uint32_t d = tmem_base + ab * 128u;
                for (int st = 0; st < nstages; ++st, ++it) {
                    const uint32_t s = it % DC_STAGES, ph = (it / DC_STAGES) & 1u;
                    mbar_wait(&full[s], ph);
                    tc_fence_after_sync();
                    const uint32_t a_base = smem_u32(a_smem + s * DC_A_BYTES);
                    const uint32_t b_base = smem_u32(b_smem + s * DC_B_BYTES);
#pragma unroll
                    for (int k16 = 0; k16 < 4; ++k16) {
                        const uint64_t ad = umma_desc_nosw(a_base + k16 * 2 * DC_A_LBO, DC_A_LBO, 128);
                        const uint64_t bd = umma_desc_nosw(b_base + k16 * 2 * lbo_b, lbo_b, 128);
                        umma_f16(d, ad, bd, idesc, (st | k16) != 0 ? 1u : 0u);
                    }
                    umma_commit(&empty[s]);
                }
                umma_commit(&acc_full[ab]);
            }
        }
    } else if (warp < 6) {
        // ================= epilogue: warps 2..5 -> TMEM lane quarters 2,3,0,1
        const int q = warp & 3;
        uint32_t acc_it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++acc_it) {
            const int nt = tile % P.n_tiles_n, pt = tile / P.n_tiles_n;
            const int tx = pt % tiles_x, ty = (pt / tiles_x) % tiles_y, img = pt / (tiles_x * tiles_y);
            const uint32_t ab = acc_it & 1u;
            mbar_wait_warp(&acc_full[ab], (acc_it >> 1) & 1u);
            tc_fence_after_sync();
            const int y = ty * DC_TILE_H + 4 * q + (lane >> 3);
            const int x = tx * DC_TILE_W + (lane & 7);
            const bool valid = (y < P.Ho) && (x < P.Wo);
            const uint32_t t0 = tmem_base + (static_cast<uint32_t>(32 * q) << 16) + ab * 128u;
#pragma unroll 1
            for (int cc = 0; cc < P.BN; cc += 32) {
                float v[32];
                tmem_ld32(t0 + cc, v);
                epi_store32<EK_NCHW>(P.epi, has_bias ? bias_s : nullptr, v, img, y, x, nt * P.BN + cc, valid);
            }
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[ab]);
        }
    } else if (warp == DC_THREADS / 32 - 1) {
        // ================= forwarder: "all gather warps have written stage s" -> generic->async proxy fence -> full[s].
        // The fence used to sit in every gather thread (MEMBAR.ALL.CTA), where it also waited for the thread's prefetched
        // offset loads of the NEXT stage, i.e. it undid the software pipelining of the gather.
        if (lane == 0) {
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x)
                for (int st = 0; st < nstages; ++st, ++it) {
                    const uint32_t s = it % DC_STAGES, ph = (it / DC_STAGES) & 1u;
                    mbar_wait(&gathered[s], ph);
                    fence_proxy_async_smem();
                    mbar_arrive(&full[s]);
                }
        }
    } else {
        // ================= gather warps (256 threads): build the A operand of each stage.
        // lane -> (pixel slot = lane/4, channel-atom pair kp = lane%4 -> atoms 2kp, 2kp+1 = 32 contiguous bytes);
        // a thread owns DC_NPX pixels per stage.  The 4 lanes of a pixel cover one full 128-byte line per corner.
        // All kernel parameters used below are copied to registers first: with two gather warps per scheduler
        // every constant-bank load / integer division inside the stage loop is exposed latency.
        const int gw = warp - 6;                      // 0 .. DC_GATHER_THREADS/32 - 1
        const int kc0 = (lane & 3) * 2;
        const int H = P.H, W = P.W, Ho = P.Ho, Wo = P.Wo, strd = P.stride, pad = P.pad, dil = P.dil;
        const int strd_w = P.stride_w, pad_w = P.pad_w, dil_w = P.dil_w;
        const int kw = P.kw, cpg = P.cpg, dg = P.dg;
        const float fH = static_cast<float>(H), fW = static_cast<float>(W);
        const long long xps = P.x_pix_stride, xrow = static_cast<long long>(W) * xps;
        const __half* const xview = P.x + P.x_ch_off;
        const long long plane = static_cast<long long>(Ho) * Wo;
        const float* const off_f = P.offset;
        const float* const msk_f = P.mask;
        const bool wide = P.x_wide != 0;

        struct Pix { int m, hb, wb; bool ok; const float* ob; const float* mb; };
        auto fetch = [&](const Pix& px, int g, int tap) -> DcnOff {
            DcnOff o;
            o.dh = o.dw = o.mk = 0.f;
            if (px.ok) {
                const float* ob = px.ob + (static_cast<long long>(g) * 2 * K + 2 * tap) * plane;
                o.dh = __ldg(ob);
                o.dw = __ldg(ob + plane);
                o.mk = msk_f ? __ldg(px.mb + (static_cast<long long>(g) * K + tap) * plane) : 1.f;
            }
            return o;
        };
        const int ixps = static_cast<int>(xps), ixrow = static_cast<int>(xrow);
        auto corner = [&](const Pix& px, int ki, int kj, const DcnOff& o) -> DcnCorner {
            DcnCorner c;
            c.off[0] = c.off[1] = c.off[2] = c.off[3] = -1;
            c.w[0] = c.w[1] = c.w[2] = c.w[3] = 0.f;
            const float h_im = static_cast<float>(px.hb + ki * dil) + o.dh;
            const float w_im = static_cast<float>(px.wb + kj * dil_w) + o.dw;
            if (px.ok && h_im > -1.f && w_im > -1.f && h_im < fH && w_im < fW) {
                const float hf = floorf(h_im), wf = floorf(w_im);
                const int hl = static_cast<int>(hf), wl = static_cast<int>(wf);
                const float lh = h_im - hf, lw = w_im - wf, hh = 1.f - lh, hw = 1.f - lw;
                c.w[0] = hh * hw * o.mk; c.w[1] = hh * lw * o.mk; c.w[2] = lh * hw * o.mk; c.w[3] = lh * lw * o.mk;
                const bool t = hl >= 0, b = hl + 1 <= H - 1, l = wl >= 0, r = wl + 1 <= W - 1;
                const int base = hl * ixrow + wl * ixps;
                c.off[0] = (t && l) ? base : -1;
                c.off[1] = (t && r) ? base + ixps : -1;
                c.off[2] = (b && l) ? base + ixrow : -1;
                c.off[3] = (b && r) ? base + ixrow + ixps : -1;
            }
            return c;
        };
        const __half* const zbuf = reinterpret_cast<const __half*>(dcn_zero32);

        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int pt = tile / P.n_tiles_n;
            const int tx = pt % tiles_x, ty = (pt / tiles_x) % tiles_y, img = pt / (tiles_x * tiles_y);
            const __half* const ximg = xview + static_cast<long long>(img) * H * xrow;
            Pix px[DC_NPX];
#pragma unroll
            for (int i = 0; i < DC_NPX; ++i) {
                px[i].m = i * (128 / DC_NPX) + gw * 8 + (lane >> 2);
                const int ho = ty * DC_TILE_H + (px[i].m >> 3), wo = tx * DC_TILE_W + (px[i].m & 7);
                px[i].ok = (ho < Ho) && (wo < Wo);
                px[i].hb = ho * strd - pad;
                px[i].wb = wo * strd_w - pad_w;
                const long long pix = static_cast<long long>(ho) * Wo + wo;
                px[i].ob = off_f + static_cast<long long>(img) * dg * 2 * K * plane + pix;
                px[i].mb = msk_f + static_cast<long long>(img) * dg * K * plane + pix;
            }
            // software pipeline: the (dh, dw, mask) triples of the NEXT stage are fetched while this one is gathered
            int g0 = (kc0 * 8) / cpg, g1 = (kc0 * 8 + 8) / cpg;
            DcnOff nxt[DC_NPX][2];
#pragma unroll
            for (int i = 0; i < DC_NPX; ++i) {
                nxt[i][0] = fetch(px[i], g0, 0);
                nxt[i][1] = (g1 != g0) ? fetch(px[i], g1, 0) : nxt[i][0];
            }
            for (int chunk = 0; chunk < nchunks; ++chunk) {
                const int ch = chunk * 64 + kc0 * 8;
                const bool two = g1 != g0;                     // cpg == 8: the two atoms belong to different groups
                const int chn = ch + 64;
                const int ng0 = (chunk + 1 < nchunks) ? chn / cpg : g0, ng1 = (chunk + 1 < nchunks) ? (chn + 8) / cpg : g1;
                int ki = 0, kj = 0;
                for (int tap = 0; tap < K; ++tap, ++it) {
                    const uint32_t s = it % DC_STAGES, ph = (it / DC_STAGES) & 1u;
                    DcnCorner cn[DC_NPX][2];
#pragma unroll
                    for (int i = 0; i < DC_NPX; ++i) {
                        cn[i][0] = corner(px[i], ki, kj, nxt[i][0]);
                        cn[i][1] = two ? corner(px[i], ki, kj, nxt[i][1]) : cn[i][0];
                    }
                    // all 16 corner loads in flight before anything is consumed
                    uint4 u[DC_NPX][2][4];
                    if (wide && !two) {
                        // the lane's two K atoms (one deformable group, 32 contiguous bytes) in ONE load per corner: the four
                        // lanes of a pixel fetch a full 128-byte line per instruction (half the L1 wavefronts of 2 x LDG.128)
#pragma unroll
                        for (int i = 0; i < DC_NPX; ++i)
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const int o = cn[i][0].off[k];
                                ldg_nc_v8(o >= 0 ? ximg + o + ch : zbuf, u[i][0][k], u[i][1][k]);
                            }
                    } else {
#pragma unroll
                        for (int i = 0; i < DC_NPX; ++i)
#pragma unroll
                            for (int a = 0; a < 2; ++a)
#pragma unroll
                                for (int k = 0; k < 4; ++k) {
                                    const int o = cn[i][a].off[k];
                                    u[i][a][k] = ldg_nc_v4(o >= 0 ? ximg + o + ch + a * 8 : zbuf);
                                }
                    }
                    // prefetch the next stage's offsets (next tap of this chunk, or tap 0 of the next chunk)
                    {
                        const bool last_tap = tap + 1 == K;
                        const int t1 = last_tap ? 0 : tap + 1;
                        const int h0 = last_tap ? ng0 : g0, h1 = last_tap ? ng1 : g1;
                        if (!(last_tap && chunk + 1 == nchunks)) {
#pragma unroll
                            for (int i = 0; i < DC_NPX; ++i) {
                                nxt[i][0] = fetch(px[i], h0, t1);
                                nxt[i][1] = (h1 != h0) ? fetch(px[i], h1, t1) : nxt[i][0];
                            }
                        }
                    }
                    if (++kj == kw) { kj = 0; ++ki; }
                    // the smem slot is needed only now
                    mbar_wait_warp(&empty[s], ph ^ 1u);
                    const uint32_t dst = smem_u32(a_smem + s * DC_A_BYTES) + kc0 * DC_A_LBO;
#pragma unroll
                    for (int i = 0; i < DC_NPX; ++i)
#pragma unroll
                        for (int a = 0; a < 2; ++a) {
                            float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                            dcn_blend8(acc, u[i][a][0], cn[i][a].w[0]);
                            dcn_blend8(acc, u[i][a][1], cn[i][a].w[1]);
                            dcn_blend8(acc, u[i][a][2], cn[i][a].w[2]);
                            dcn_blend8(acc, u[i][a][3], cn[i][a].w[3]);
                            const uint4 r = make_uint4(pack_h2(acc[0], acc[1]), pack_h2(acc[2], acc[3]), pack_h2(acc[4], acc[5]),
                                                       pack_h2(acc[6], acc[7]));
                            sts_v4(dst + a * DC_A_LBO + px[i].m * 16, r);
                        }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&gathered[s]);
                }
                g0 = ng0;
                g1 = ng1;
            }
        }
    }

    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 256);
}

}  // namespace eb
