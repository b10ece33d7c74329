// conv_pair.cuh — 3x3 (pad 1) and 1x1 convolutions as an implicit GEMM issued by CTA PAIRS (tcgen05 cta_group::2); weights
// resident in shared memory when they fit (K * BN <= 147456 elements per CTA pair, e.g. 128 -> 128 3x3), streamed otherwise.
//
// Why (all measured on B200, tools/mma_rate.py + tools/one_conv.py, profiles/r01_one_conv_*.log):
//   * back-to-back tcgen05.mma run at their floor (64 cycles for 128x128x16) in every layout, so the single-CTA
//     kernels were never short of operand bandwidth: they lost the tensor pipe to the ISSUE path (15 dependent
//     instructions per MMA from a lane-0 branch, a proxy fence in the issuing thread, 18 weight-stage handshakes per
//     tile) and to the LSU (cp.async / st.global wavefronts of loaders and epilogue);
//   * here the two CTAs of a cluster each own one 16x16 pixel tile (M = 2 x 128 rows per MMA) and HALF of the output
//     channels of the weight matrix (B operand split along N), and each CTA's half of the weights stays RESIDENT in
//     shared memory for the whole kernel: no weight ring, no per-stage weight handshake, no L2 weight traffic after
//     the prologue;
//   * activations arrive by TMA: one 5-D box {8 channels, 18 x, 18 y, 4 K-atoms, 1 image} per 32-channel stage lands
//     exactly in the K-atom-plane layout of conv_igemm.cuh (nine taps = nine start addresses), zero-filled outside the
//     image by the copy engine, counted on the even CTA's mbarrier by both CTAs - no loader warps, no LSU traffic, no
//     generic->async proxy fence;
//   * the fp16 NHWC output leaves through TMA as well: each epilogue warp stages its 32 pixels x 32 channels in a private
//     2 KB buffer (64-byte swizzle, conflict-free) and one lane issues a box store - full 64-byte segments per pixel
//     instead of 32 scattered 16-byte st.global per instruction (the epilogue's LSU wavefronts cost 4K cycles per tile);
//   * the MMA warp runs converged and elects one lane per instruction, descriptors live in uniform registers;
//   * layers whose weights do not fit (Cin = 256) use the same kernel with RESIDENT = false: each CTA's half of the weights
//     of a 32-channel chunk (36 KB) travels with the activation stage as a second TMA box on the same mbarrier.
// Only the even CTA issues MMAs; completion is multicast to both CTAs' mbarriers; the odd CTA's epilogue warps signal
// "accumulator drained" to the even CTA through the cluster shared-memory window.
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "conv_igemm.cuh"
#include "epilogue.cuh"

namespace eb {

constexpr int CP_CH = 32;                                   // channels per activation stage
constexpr int CP_A_STAGES = 3;
constexpr int CP_RP = CV_TILE + 2;                          // halo tile edge
constexpr int CP_PLANE_BYTES = CP_RP * CP_RP * 16;          // 5184: one K atom (8 channels) of every halo pixel, dense (TMA box order)
constexpr int CP_A_STAGE_BYTES = 4 * CP_PLANE_BYTES;        // 20736
constexpr int CP_W_BYTES = 147456;                          // resident weights per CTA: (BN/2) x K fp16
constexpr int CP_MAX_WGROUPS = 8;
constexpr int CP_THREADS = 320;                             // warp 0 producer, warp 1 MMA, warps 2-9 epilogue
constexpr int CP_OUT_STAGE_BYTES = 32 * 64;                 // per epilogue warp: 32 pixels x 32 fp16 channels
constexpr int CP_W_STAGE_BYTES = 9 * 4 * 64 * 16;           // streamed mode: weights of one chunk, BN/2 <= 64 rows
constexpr int CP_SMEM_BYTES = CP_W_BYTES + 8 * CP_OUT_STAGE_BYTES + CP_A_STAGES * CP_A_STAGE_BYTES + 128 * 4 + 256;
constexpr int CP_SMEM_BYTES_STREAM = 8 * CP_OUT_STAGE_BYTES + CP_A_STAGES * (CP_A_STAGE_BYTES + CP_W_STAGE_BYTES) + 128 * 4 + 256;
// 1x1 layers: no halo, 64 channels per stage (eight K atoms of a 16x16 tile = 32 KB) + 8 KB of streamed weights
constexpr int CP1_A_STAGE_BYTES = 8 * CV_TILE * CV_TILE * 16;
constexpr int CP1_W_STAGE_BYTES = 4 * 2 * 64 * 16;
constexpr int CP_SMEM_BYTES_1X1 = 8 * CP_OUT_STAGE_BYTES + CP_A_STAGES * (CP1_A_STAGE_BYTES + CP1_W_STAGE_BYTES) + 128 * 4 + 256;

struct PairParams {
    ConvParams c;
    CUtensorMap tmap[2];        // one per source: dims {8 ch, W, H, pix_stride/8 atoms, images}, box {8, 18, 18, 4, 1}
    CUtensorMap tmap_w;         // streamed weights: packed array as rows of 256 fp16, box = one chunk stage of one CTA
    CUtensorMap tmap_out;       // fp16 NHWC output: dims {pix_stride, W, H, N}, box {32 ch, 8 x, 4 y, 1}, 64-byte swizzle
    int tma_out;                // 1: out16 leaves through tmap_out
};

template <int EK, bool TMA_OUT, bool RESIDENT, int TAPS = 9>
__global__ void __launch_bounds__(CP_THREADS, 1) conv_pair_kernel(const __grid_constant__ PairParams PP) {
    const ConvParams& P = PP.c;
    extern __shared__ __align__(1024) uint8_t smem[];
    static_assert(TAPS == 9 || (TAPS == 1 && !RESIDENT), "1x1 layers stream their weights");
    constexpr int RP = TAPS == 9 ? CP_RP : CV_TILE;           // edge of the activation tile in shared memory
    constexpr int CH = TAPS == 9 ? CP_CH : 64;                // channels per stage
    constexpr int KSTEPS = CH / 16;                           // K16 steps per tap and stage
    constexpr int NSTEP = TAPS * KSTEPS;                      // (tap, K16) steps per stage = MMAs per 128-pixel half
    constexpr int PLANE_BYTES = RP * RP * 16;
    constexpr int A_STAGE_BYTES = (CH / 8) * PLANE_BYTES;
    constexpr int W_STAGE_BYTES = NSTEP * 2 * 64 * 16;        // streamed weights of one stage at BN/2 = 64 rows
    // resident: [weights 144 KB][output staging 16 KB][3 activation stages]; streamed: [output staging][3 x (activations, weights)]
    constexpr int STAGE_STRIDE = RESIDENT ? A_STAGE_BYTES : A_STAGE_BYTES + W_STAGE_BYTES;
    uint8_t* w_smem = smem;
    uint8_t* o_smem = smem + (RESIDENT ? CP_W_BYTES : 0);    // 8 x 2 KB output staging (1024-byte aligned)
    uint8_t* a_smem = o_smem + 8 * CP_OUT_STAGE_BYTES;
    float* bias_s = reinterpret_cast<float*>(a_smem + CP_A_STAGES * STAGE_STRIDE);
    uint64_t* bars = reinterpret_cast<uint64_t*>(bias_s + 128);
    uint64_t* a_full = bars;                         // [CP_A_STAGES]  even CTA: both CTAs' TMA boxes (2 arrivals + bytes)
    uint64_t* a_empty = a_full + CP_A_STAGES;        // [CP_A_STAGES]  multicast commit
    uint64_t* w_full = a_empty + CP_A_STAGES;        // [CP_MAX_WGROUPS]
    uint64_t* acc_full = w_full + CP_MAX_WGROUPS;    // [2]            multicast commit
    uint64_t* acc_empty = acc_full + 2;              // [2]            even CTA only: 8 local + 8 remote epilogue warps
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;

    const int tiles_x = (P.W + CV_TILE - 1) / CV_TILE;
    const int tiles_x2 = (tiles_x + 1) / 2;
    const int tiles_y = (P.H + CV_TILE - 1) / CV_TILE;
    const int total_pt = P.N * tiles_y * tiles_x2;           // pair tiles (two horizontally adjacent 16x16 tiles)
    const int cin = P.src[0].C + (P.nsrc > 1 ? P.src[1].C : 0);
    const int nchunks = cin / CH;
    const int half = P.BN / 2;                               // output channels (B rows) held by this CTA
    const uint32_t lbo_b = static_cast<uint32_t>(half) * 16u;
    const uint32_t stage_w_bytes = static_cast<uint32_t>(NSTEP) * 2u * lbo_b;     // weights of one stage (CH channels x TAPS)
    const int wgroups = nchunks < CP_MAX_WGROUPS ? nchunks : CP_MAX_WGROUPS;
    const int cpg = (nchunks + wgroups - 1) / wgroups;       // chunks per weight group

    // clusters are partitioned over the n-tiles so that each keeps ONE weight slice resident
    const int cluster_id = blockIdx.x >> 1, nclusters = gridDim.x >> 1;
    const int nt = cluster_id % P.n_tiles_n;
    const int cpn = nclusters / P.n_tiles_n;                 // clusters per n-tile (host guarantees >= 1)
    const int ci = cluster_id / P.n_tiles_n;
    const bool active = ci < cpn && ci < total_pt;

    // ---- one-time setup
    const bool has_bias = P.epi.bias != nullptr;
    if (has_bias && threadIdx.x < P.BN) bias_s[threadIdx.x] = P.epi.bias[nt * P.BN + threadIdx.x];
    if (threadIdx.x == 0) {
        for (int i = 0; i < CP_A_STAGES; ++i) { mbar_init(&a_full[i], 2); mbar_init(&a_empty[i], 1); }
        for (int i = 0; i < CP_MAX_WGROUPS; ++i) mbar_init(&w_full[i], leader ? 2 : 1);     // resident mode only
        for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 16); }
        fence_barrier_init();
        tma_prefetch_desc(&PP.tmap[0]);
        if (P.nsrc > 1) tma_prefetch_desc(&PP.tmap[1]);
        if (TMA_OUT) tma_prefetch_desc(&PP.tmap_out);
        if (!RESIDENT) tma_prefetch_desc(&PP.tmap_w);
    }
    if (warp == 0) tmem_alloc_pair(tmem_slot, 512);
    tc_fence_before_sync();
    __syncthreads();
    cluster_sync_all();                                      // both CTAs' barriers and TMEM exist before any remote traffic
    tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    // Programmatic dependent launch: the next kernel of the stream may begin its prologue (barriers, TMEM, weights) on SMs
    // this grid has already left - the tail of a 6.5-round launch leaves half of them idle.  Everything above and the weight
    // copies below touch only constants; activations, residuals and outputs wait for the predecessor (pdl_wait).
    pdl_trigger();
    if (!(active && warp == 0 && lane == 0)) pdl_wait();

    if (active) {
        if (warp == 0) {
            if (lane == 0) {
                // ================= producer.  Weights: this CTA's half of n-tile nt, once, in consumption order.
                const uint8_t* w = reinterpret_cast<const uint8_t*>(P.wpack) +
                                   (static_cast<size_t>(nt) * 2 + rank) * nchunks * stage_w_bytes;
                for (int g = 0; RESIDENT && g < wgroups; ++g) {
                    const int c0 = g * cpg, c1 = (c0 + cpg < nchunks) ? c0 + cpg : nchunks;
                    if (c1 <= c0) { mbar_arrive(&w_full[g]); continue; }
                    mbar_arrive_expect_tx(&w_full[g], static_cast<uint32_t>(c1 - c0) * stage_w_bytes);
                    for (int c = c0; c < c1; ++c)
                        bulk_g2s(w_smem + static_cast<size_t>(c) * stage_w_bytes, w + static_cast<size_t>(c) * stage_w_bytes,
                                 stage_w_bytes, &w_full[g]);
                }
                pdl_wait();
                // Activations: one TMA box per stage into this CTA, bytes counted on the even CTA's a_full.
                uint32_t a_it = 0;
                bool first = RESIDENT;
                const int w_rows = static_cast<int>(stage_w_bytes / 512u);           // streamed: rows of 256 fp16 per chunk stage
                const int w_row0 = (nt * 2 + static_cast<int>(rank)) * nchunks * w_rows;
                for (int t = ci; t < total_pt; t += cpn) {
                    const int tx = (t % tiles_x2) * 2 + static_cast<int>(rank), ty = (t / tiles_x2) % tiles_y;
                    const int img = t / (tiles_x2 * tiles_y);
                    for (int c = 0; c < nchunks; ++c, ++a_it) {
                        if (first && !leader && c % cpg == 0) { mbar_wait(&w_full[c / cpg], 0); mbar_arrive_remote(&w_full[c / cpg], 0); }
                        int s = 0, ch = c * CH;
                        if (P.nsrc > 1 && ch >= P.src[0].C) { s = 1; ch -= P.src[0].C; }
                        const ConvSrc& S = P.src[s];
                        const int simg = (img / S.div) * S.mul + (img % S.div) * S.keep + S.add;
                        const uint32_t as = a_it % CP_A_STAGES, aph = (a_it / CP_A_STAGES) & 1u;
                        mbar_wait(&a_empty[as], aph ^ 1u);
                        const bool skip = (P.dbg & 16) && a_it >= CP_A_STAGES;           // profiling: reuse stale stages
                        const uint32_t bytes = skip ? 0u : static_cast<uint32_t>(A_STAGE_BYTES) + (RESIDENT ? 0u : stage_w_bytes);
                        if (leader) mbar_arrive_expect_tx(&a_full[as], bytes);
                        else mbar_arrive_expect_tx_remote(&a_full[as], bytes, 0);
                        if (!skip) {
                            tma_load_5d_pair(a_smem + as * STAGE_STRIDE, &PP.tmap[s], &a_full[as], 0, tx * CV_TILE - (TAPS == 9),
                                             ty * CV_TILE - (TAPS == 9), (S.ch_off + ch) >> 3, simg);
                            if (!RESIDENT)
                                tma_load_2d_pair(a_smem + as * STAGE_STRIDE + A_STAGE_BYTES, &PP.tmap_w, &a_full[as], 0,
                                                 w_row0 + c * w_rows);
                        }
                    }
                    first = false;
                }
            }
        } else if (warp == 1) {
            if (leader) {
                // ================= MMA issuer (even CTA): M = 256 rows (128 per CTA), N = BN, K = 16 per instruction.
                // All 32 lanes run the loops (uniform control flow), one elected lane issues.
                const uint32_t idesc = umma_idesc_f16(256, P.BN, P.epi.bf16 ? 1u : 0u);
                const uint32_t w_lo0 = umma_desc_lo(smem_u32(w_smem), lbo_b);
                const uint32_t a_hi = umma_desc_hi(RP * 16), b_hi = umma_desc_hi(128);
                const uint32_t b_step = (2u * lbo_b) >> 4;                 // one K16 step of the resident weights
                // Waits are software-pipelined: everything stage n+1 needs (its TMA boxes; at a tile boundary the drained
                // accumulator; on the first tile the weight group) is awaited in the MIDDLE of issuing stage n, while ~20 MMAs
                // are still queued - the barrier round trip no longer leaves the tensor pipe idle between stages.
                uint32_t a_it = 0, acc_it = 0;
                auto wait_stage = [&](int c, uint32_t ait, uint32_t accit, bool first_tile) {
                    if (c == 0) mbar_wait_cluster(&acc_empty[accit & 1u], ((accit >> 1) & 1u) ^ 1u);
                    if (RESIDENT && first_tile && c % cpg == 0) mbar_wait_cluster(&w_full[c / cpg], 0);
                    mbar_wait_cluster(&a_full[ait % CP_A_STAGES], (ait / CP_A_STAGES) & 1u);
                };
                if (ci < total_pt) wait_stage(0, 0, 0, true);
                for (int t = ci; t < total_pt; t += cpn, ++acc_it) {
                    const uint32_t ab = acc_it & 1u;
                    const bool first = t == ci;
                    const uint32_t d0 = tmem_base + ab * 256u;
                    for (int c = 0; c < nchunks; ++c, ++a_it) {
                        const uint32_t as = a_it % CP_A_STAGES;
                        tc_fence_after_sync();
                        const uint32_t a_lo0 = umma_desc_lo(smem_u32(a_smem + as * STAGE_STRIDE), PLANE_BYTES);
                        const uint32_t b_lo0 = RESIDENT ? w_lo0 + static_cast<uint32_t>(c) * NSTEP * b_step
                                                        : umma_desc_lo(smem_u32(a_smem + as * STAGE_STRIDE + A_STAGE_BYTES), lbo_b);
                        const bool skip = (P.dbg & 32) != 0;
                        constexpr int SPLIT = (NSTEP + 1) / 2 + (TAPS == 9 ? 1 : 0);      // first part: 10 of 18 (tap, K16) steps
                        if (!skip && elect_one()) {
                            uint32_t acc = c != 0 ? 1u : 0u;
#pragma unroll
                            for (int i = 0; i < SPLIT; ++i) {
                                const int tp = i / KSTEPS, h = i % KSTEPS;
                                const int ki = TAPS == 9 ? tp / 3 : 0, kj = TAPS == 9 ? tp % 3 : 0;
                                const uint32_t a_lo = a_lo0 + (ki * RP + kj) + h * (2 * PLANE_BYTES / 16);
                                const uint32_t b_lo = b_lo0 + i * b_step;
                                umma_f16_lohi<2>(d0, a_lo, a_hi, b_lo, b_hi, idesc, acc);
                                umma_f16_lohi<2>(d0 + 128u, a_lo + 8, a_hi, b_lo, b_hi, idesc, acc);
                                acc = 1u;
                            }
                        }
                        __syncwarp();
                        // requirements of the next stage (possibly the first stage of the next tile)
                        if (c + 1 < nchunks) wait_stage(c + 1, a_it + 1, acc_it, first);
                        else if (t + cpn < total_pt) wait_stage(0, a_it + 1, acc_it + 1, false);
                        if (elect_one()) {
                            if (!skip) {
#pragma unroll
                                for (int i = SPLIT; i < NSTEP; ++i) {
                                    const int tp = i / KSTEPS, h = i % KSTEPS;
                                    const int ki = TAPS == 9 ? tp / 3 : 0, kj = TAPS == 9 ? tp % 3 : 0;
                                    const uint32_t a_lo = a_lo0 + (ki * RP + kj) + h * (2 * PLANE_BYTES / 16);
                                    const uint32_t b_lo = b_lo0 + i * b_step;
                                    umma_f16_lohi<2>(d0, a_lo, a_hi, b_lo, b_hi, idesc, 1u);
                                    umma_f16_lohi<2>(d0 + 128u, a_lo + 8, a_hi, b_lo, b_hi, idesc, 1u);
                                }
                            }
                            umma_commit_pair(&a_empty[as], 3);
                            if (c == nchunks - 1) umma_commit_pair(&acc_full[ab], 3);
                        }
                        __syncwarp();
                    }
                }
            }
        } else {
            // ================= epilogue: 8 warps per CTA (TMEM lane quarter = warp % 4), each CTA drains its own 128 lanes
            const int q = warp & 3;
            const int sub = (warp - 2) >> 2;
            uint8_t* stage = o_smem + (warp - 2) * CP_OUT_STAGE_BYTES;
            // staging row = lane (pixel), four 16-byte units XOR-swizzled like CU_TENSOR_MAP_SWIZZLE_64B: unit ^= (row >> 1) & 3
            const uint32_t st_row = smem_u32(stage) + lane * 64;
            const uint32_t st_x = ((lane >> 1) & 3) * 16;
            uint32_t acc_it = 0;
            for (int t = ci; t < total_pt; t += cpn, ++acc_it) {
                const int tx = (t % tiles_x2) * 2 + static_cast<int>(rank), ty = (t / tiles_x2) % tiles_y;
                const int img = t / (tiles_x2 * tiles_y);
                const uint32_t ab = acc_it & 1u;
                const int y0 = ty * CV_TILE + 4 * q, x0 = tx * CV_TILE + 8 * sub;
                const int y = y0 + (lane >> 3);
                const int x = x0 + (lane & 7);
                const bool valid = (y < P.H) && (x < P.W) && !(P.dbg & 1);
                const bool box_ok = (y0 < P.H) && (x0 < P.W) && !(P.dbg & 1);          // warp-uniform
                float4 rpre_a[8], rpre_b[8];
                const bool pre_ok = !(P.dbg & 4) && ((EK == EK_F32 && P.epi.res32 != nullptr && P.epi.f32_blocked != 0) ||
                                                     (EK == EK_PLAIN && P.epi.res16 != nullptr));
                auto prefetch = [&](int c0, float4 (&r)[8]) {
                    if (EK == EK_F32) epi_prefetch_res32_blocked(P.epi, img, y, x, c0, valid, r);
                    else epi_prefetch_res16(P.epi, img, y, x, c0, valid, r);
                };
                if ((EK == EK_F32 || EK == EK_PLAIN) && pre_ok) prefetch(nt * P.BN, rpre_a);
                mbar_wait_warp(&acc_full[ab], (acc_it >> 1) & 1u);
                tc_fence_after_sync();
                const uint32_t t0 = tmem_base + (static_cast<uint32_t>(32 * q) << 16) + ab * 256u + sub * 128u;
                auto do_chunk = [&](int cc, const float4* pre) {
                    float v[32];
                    tmem_ld32(t0 + cc, v);
                    epi_store32<EK, TMA_OUT>(P.epi, has_bias ? bias_s - nt * P.BN : nullptr, v, img, y, x, nt * P.BN + cc, valid, pre);
                    if (TMA_OUT && EK == EK_PIXSHUF) {
                        // PixelShuffle(2): conv channel 4k + 2i + j of pixel (y, x) is output channel k of pixel (2y+i, 2x+j)
                        // (edvr_arch.py:351,410-411).  Staging = the 8 x 16 output pixels of this warp, 8 channels (16 B) each,
                        // in the box order {8 ch, 16 x, 8 y} of the output tensor map.
                        if (lane == 0) bulk_wait_group_read0();
                        __syncwarp();
                        const uint32_t sp = smem_u32(stage) + ((2 * (lane >> 3)) * 16 + 2 * (lane & 7)) * 16;
#pragma unroll
                        for (int i = 0; i < 2; ++i)
#pragma unroll
                            for (int j = 0; j < 2; ++j) {
                                const int sidx = 2 * i + j;
                                sts_v4(sp + (i * 16 + j) * 16,
                                       make_uint4(pack_h2(v[sidx], v[4 + sidx]), pack_h2(v[8 + sidx], v[12 + sidx]),
                                                  pack_h2(v[16 + sidx], v[20 + sidx]), pack_h2(v[24 + sidx], v[28 + sidx])));
                            }
                        fence_proxy_async_smem();
                        __syncwarp();
                        if (lane == 0 && box_ok) {
                            tma_store_4d(&PP.tmap_out, stage, P.epi.out16_ch_off + ((nt * P.BN + cc) >> 2), 2 * x0, 2 * y0, img);
                            bulk_commit_group();
                        }
                    } else if (TMA_OUT) {
                        if (lane == 0) bulk_wait_group_read0();          // the previous box has been read out of the staging buffer
                        __syncwarp();
                        if (EK == EK_PLAIN && P.epi.bf16) {            // training step: bf16 activations
#pragma unroll
                            for (int u = 0; u < 4; ++u)
                                sts_v4(st_row + ((u * 16) ^ st_x),
                                       make_uint4(pack_bf2(v[u * 8 + 0], v[u * 8 + 1]), pack_bf2(v[u * 8 + 2], v[u * 8 + 3]),
                                                  pack_bf2(v[u * 8 + 4], v[u * 8 + 5]), pack_bf2(v[u * 8 + 6], v[u * 8 + 7])));
                        } else {
#pragma unroll
                            for (int u = 0; u < 4; ++u)
                                sts_v4(st_row + ((u * 16) ^ st_x),
                                       make_uint4(pack_h2(v[u * 8 + 0], v[u * 8 + 1]), pack_h2(v[u * 8 + 2], v[u * 8 + 3]),
                                                  pack_h2(v[u * 8 + 4], v[u * 8 + 5]), pack_h2(v[u * 8 + 6], v[u * 8 + 7])));
                        }
                        fence_proxy_async_smem();
                        __syncwarp();
                        if (lane == 0 && box_ok) {
                            tma_store_4d(&PP.tmap_out, stage, P.epi.out16_ch_off + nt * P.BN + cc, x0, y0, img);
                            bulk_commit_group();
                        }
                    }
                
                };
                const int bn_epi = (P.dbg & 4) ? 0 : P.BN;
                if ((EK == EK_F32 || EK == EK_PLAIN) && pre_ok) {
                    // residual stream (blocked fp32 of the trunk, fp16 elsewhere): chunk c+1's residual is in flight while chunk c
                    // is processed (two static register buffers; the first one was requested before the accumulator wait)
#pragma unroll 1
                    for (int cc = 0; cc < bn_epi; cc += 64) {
                        if (cc + 32 < bn_epi) prefetch(nt * P.BN + cc + 32, rpre_b);
                        do_chunk(cc, rpre_a);
                        if (cc + 32 < bn_epi) {
                            if (cc + 64 < bn_epi) prefetch(nt * P.BN + cc + 64, rpre_a);
                            do_chunk(cc + 32, rpre_b);
                        }
                    }
                } else {
#pragma unroll 1
                    for (int cc = 0; cc < bn_epi; cc += 32) do_chunk(cc, nullptr);
                }
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) { if (leader) mbar_arrive(&acc_empty[ab]); else mbar_arrive_remote(&acc_empty[ab], 0); }
            }
            if (TMA_OUT && lane == 0) bulk_wait_group0();        // all output boxes written before the CTA retires
        }
    }

    // ---- teardown: nobody leaves while the peer may still read this CTA's shared memory or signal its barriers
    tc_fence_before_sync();
    __syncthreads();
    cluster_sync_all();
    if (warp == 0) tmem_dealloc_pair(tmem_base, 512);
}

}  // namespace eb
