// conv_igemm.cuh — dense 3x3 (pad 1) / 1x1 convolution as an implicit GEMM on tcgen05.
//
// Replaces every cuDNN-dispatched nn.Conv2d on the EDVR path
// (/root/reference/basicsr/models/archs/edvr_arch.py:36-66,138-155,232-244,327-353 and
//  arch_util.py:84-95) for NHWC fp16 activations, fp32 accumulation in TMEM.
//
// CTA tile  : 16x16 output pixels (two M=128 MMAs of 16 rows x 8 pixels) x BN<=128 channels.
// A operand : the (16+2)x(16+2) input halo of one 64-channel chunk is loaded ONCE into
//             shared memory as 8 planes of 16-byte K atoms (common.cuh layout); the nine
//             taps are nine start addresses inside it, so activations cross L2->SM once
//             per chunk instead of nine times.
// B operand : weights pre-packed on the host in consumption order
//             [n_tile][chunk][tap][kc=8][BN][8] fp16, streamed by 1-D bulk async copies.
// Pipeline  : warp 0 B-producer | warp 1 MMA issuer (converged warp, elected lane) | warps 2-5 A-producers
//             (cp.async with zero-fill, completion tracked by the mbarrier, so a whole chunk is in flight per
//             SM) | warps 6-13 epilogue (one 16x8 half of the tile each) | warp 14 forwarder (generic->async
//             proxy fence between the cp.async fills and the MMA reads); mbarrier rings; 2 x 256 TMEM columns
//             so that the epilogue of tile i overlaps the MMAs of tile i+1; persistent CTAs.
// Since the CTA-pair kernel (conv_pair.cuh) took over every 3x3 / 1x1 layer with Cin % 64 == 0, this kernel is the
// fallback (no tensor-map support, EDVR_B200_CONV_PAIR=0) and the A/B partner in the tests.
#pragma once
#include "common.cuh"
#include "epilogue.cuh"

namespace eb {

constexpr int CV_TILE = 16;
constexpr int CV_A_BUFS = 3;
constexpr int CV_B_STAGES = 5;
constexpr int CV_PLANE_BYTES = 325 * 16;              // >= 18*18*16, odd # of 16B units
constexpr int CV_A_BUF_BYTES = 8 * CV_PLANE_BYTES;    // 41600
constexpr int CV_B_STAGE_BYTES = 128 * 128;           // BN(<=128) rows x 64 ch x 2 B
constexpr int CV_MAX_COUT = 512;
constexpr int CV_THREADS = 480;          // + warp 14: forwarder (proxy fence between the cp.async loaders and the MMA issuer)
constexpr int CV_SMEM_BYTES = CV_A_BUFS * CV_A_BUF_BYTES + CV_B_STAGES * CV_B_STAGE_BYTES +
                              CV_MAX_COUT * 4 + 256;

struct ConvSrc {
    const __half* ptr;
    int C;            // channels consumed from this source (multiple of 64)
    int pix_stride;   // elements between pixels
    int ch_off;       // first channel
    // image index of accumulator image n:  (n / div) * mul + (n % div) * keep + add
    int div, mul, keep, add;
};

struct ConvParams {
    ConvSrc src[2];
    int nsrc;
    int N, H, W;      // accumulator grid (== input grid; stride handled by the epilogue)
    int taps;         // 9 or 1
    int BN;           // channels per n-tile (multiple of 32, <= 128)
    int n_tiles_n;    // number of n-tiles; packed Cout = BN * n_tiles_n
    const __half* wpack;
    EpiParams epi;
    unsigned long long* stats;   // optional [gridDim.x][16] cycle counters (profiling builds of the call only)
    int dbg;                     // profiling only (results become wrong): 1 no epilogue global memory, 4 no epilogue at all,
                                 // 8 no weight copies after the first ring fill, 16 same for activations, 32 no MMAs
};

template <int HALO>
__device__ __forceinline__ void conv_load_halo(const ConvParams& P, int chunk, int img, int ty,
                                               int tx, uint32_t abuf_saddr, int tid) {
    constexpr int RP = CV_TILE + 2 * HALO;
    constexpr int NPIX = RP * RP;
    // which source does this 64-channel chunk come from?
    int s = 0, ch = chunk * 64;
    if (P.nsrc > 1 && ch >= P.src[0].C) { s = 1; ch -= P.src[0].C; }
    const ConvSrc& S = P.src[s];
    const int simg = (img / S.div) * S.mul + (img % S.div) * S.keep + S.add;
    const int kc = tid & 7;                       // 16-byte K atom of this thread; 8 lanes = 128 contiguous bytes
    const __half* base = S.ptr + S.ch_off + ch + kc * 8;
    const __half* img_base = base + static_cast<size_t>(simg) * P.H * P.W * S.pix_stride;
    const int y0 = ty * CV_TILE - HALO, x0 = tx * CV_TILE - HALO;
    const int H = P.H, W = P.W, ps = S.pix_stride;
    uint32_t dst = abuf_saddr + kc * CV_PLANE_BYTES + (tid >> 3) * 16;
    int y = (tid >> 3) / RP, x = (tid >> 3) - y * RP;       // 16 pixels per step of the 128 threads
#pragma unroll 4
    for (int p = tid >> 3; p < NPIX; p += 16) {
        const int gy = y0 + y, gx = x0 + x;
        const bool in = (gy >= 0) & (gy < H) & (gx >= 0) & (gx < W);
        const __half* g = in ? img_base + (static_cast<size_t>(gy) * W + gx) * ps : base;
        cp_async16_zfill(dst, g, in ? 16u : 0u);
        dst += 16 * 16;
        x += 16;
        if (x >= RP) { x -= RP; ++y; }
    }
}

template <int HALO, int EK>
__global__ void __launch_bounds__(CV_THREADS, 1) conv_igemm_kernel(const ConvParams P) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* a_smem = smem;
    uint8_t* b_smem = smem + CV_A_BUFS * CV_A_BUF_BYTES;
    float* bias_s = reinterpret_cast<float*>(b_smem + CV_B_STAGES * CV_B_STAGE_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(bias_s + CV_MAX_COUT);
    uint64_t* a_full = bars;                                 // [CV_A_BUFS]
    uint64_t* a_empty = bars + CV_A_BUFS;                    // [CV_A_BUFS]
    uint64_t* b_full = bars + 2 * CV_A_BUFS;                 // [CV_B_STAGES]
    uint64_t* b_empty = b_full + CV_B_STAGES;                // [CV_B_STAGES]
    uint64_t* a_ready = b_empty + CV_B_STAGES;               // [CV_A_BUFS]  forwarder -> MMA issuer
    uint64_t* acc_full = a_ready + CV_A_BUFS;                // [2]
    uint64_t* acc_empty = acc_full + 2;                // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    constexpr int RP = CV_TILE + 2 * HALO;

    const int tiles_x = (P.W + CV_TILE - 1) / CV_TILE;
    const int tiles_y = (P.H + CV_TILE - 1) / CV_TILE;
    const int total_tiles = P.N * tiles_y * tiles_x * P.n_tiles_n;
    const int cin = P.src[0].C + (P.nsrc > 1 ? P.src[1].C : 0);
    const int nchunks = cin / 64;
    const uint32_t b_bytes = static_cast<uint32_t>(P.BN) * 128u;

    // ---- one-time setup
    const int cout_packed = P.BN * P.n_tiles_n;
    const bool has_bias = P.epi.bias != nullptr;   // host guarantees cout_packed <= CV_MAX_COUT then
    if (has_bias)
        for (int i = threadIdx.x; i < cout_packed; i += blockDim.x) bias_s[i] = P.epi.bias[i];
    if (threadIdx.x == 0) {
        for (int i = 0; i < CV_A_BUFS; ++i) { mbar_init(&a_full[i], 128); mbar_init(&a_empty[i], 1); mbar_init(&a_ready[i], 1); }
        for (int i = 0; i < CV_B_STAGES; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 8); }
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= B producer: stream packed weights, one stage per (chunk, tap)
        if (lane == 0) {
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int nt = tile % P.n_tiles_n;
                const uint8_t* w = reinterpret_cast<const uint8_t*>(P.wpack) +
                                   static_cast<size_t>(nt) * nchunks * P.taps * b_bytes;
                for (int st = 0; st < nchunks * P.taps; ++st, ++it) {
                    const uint32_t s = it % CV_B_STAGES, ph = (it / CV_B_STAGES) & 1u;
                    mbar_wait(&b_empty[s], ph ^ 1u);
                    if ((P.dbg & 8) && it >= CV_B_STAGES) { mbar_arrive(&b_full[s]); continue; }
                    mbar_arrive_expect_tx(&b_full[s], b_bytes);
                    bulk_g2s(b_smem + s * CV_B_STAGE_BYTES, w + static_cast<size_t>(st) * b_bytes,
                             b_bytes, &b_full[s]);
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer: the whole warp runs the loops (uniform control flow), one elected lane issues, so the
        // descriptors stay in uniform registers (see common.cuh, "lean issue path")
        const uint32_t idesc = umma_idesc_f16(128, P.BN);
        const uint32_t lbo_b = static_cast<uint32_t>(P.BN) * 16u;
        const uint32_t a_hi = umma_desc_hi(RP * 16), b_hi = umma_desc_hi(128);
        uint32_t a_it = 0, b_it = 0, acc_it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++acc_it) {
            const uint32_t ab = acc_it & 1u;
            mbar_wait(&acc_empty[ab], ((acc_it >> 1) & 1u) ^ 1u);
            tc_fence_after_sync();
            for (int c = 0; c < nchunks; ++c, ++a_it) {
                const uint32_t as = a_it % CV_A_BUFS, aph = (a_it / CV_A_BUFS) & 1u;
                mbar_wait(&a_ready[as], aph);
                tc_fence_after_sync();
                const uint32_t a_lo0 = umma_desc_lo(smem_u32(a_smem + as * CV_A_BUF_BYTES), CV_PLANE_BYTES);
                for (int t = 0; t < P.taps; ++t, ++b_it) {
                    const uint32_t bs = b_it % CV_B_STAGES, bph = (b_it / CV_B_STAGES) & 1u;
                    mbar_wait(&b_full[bs], bph);
                    tc_fence_after_sync();
                    const uint32_t b_lo0 = umma_desc_lo(smem_u32(b_smem + bs * CV_B_STAGE_BYTES), lbo_b);
                    const int ki = HALO ? t / 3 : 0, kj = HALO ? t % 3 : 0;
                    if (elect_one()) {
                        if (!(P.dbg & 32)) {
#pragma unroll
                            for (int k16 = 0; k16 < 4; ++k16) {
                                const uint32_t a_lo = a_lo0 + (ki * RP + kj) + k16 * (2 * CV_PLANE_BYTES / 16);
                                const uint32_t b_lo = b_lo0 + k16 * ((2u * lbo_b) >> 4);
                                const uint32_t acc = (c | t | k16) != 0 ? 1u : 0u;
                                umma_f16_lohi<1>(tmem_base + ab * 256u, a_lo, a_hi, b_lo, b_hi, idesc, acc);
                                umma_f16_lohi<1>(tmem_base + ab * 256u + 128u, a_lo + 8, a_hi, b_lo, b_hi, idesc, acc);
                            }
                        }
                        umma_commit(&b_empty[bs]);
                        if (t == P.taps - 1) umma_commit(&a_empty[as]);
                        if (t == P.taps - 1 && c == nchunks - 1) umma_commit(&acc_full[ab]);
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp == 14) {
        // ================= forwarder: "chunk landed" (cp.async, generic proxy) -> fence.proxy.async -> a_ready.  In the issuing
        // thread this fence drained the MMA queue at every chunk.
        if (lane == 0) {
            uint32_t a_it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x)
                for (int c = 0; c < nchunks; ++c, ++a_it) {
                    const uint32_t as = a_it % CV_A_BUFS, aph = (a_it / CV_A_BUFS) & 1u;
                    mbar_wait(&a_full[as], aph);
                    fence_proxy_async_smem();
                    mbar_arrive(&a_ready[as]);
                }
        }
    } else if (warp < 6) {
        // ================= A producers (128 threads): halo tile of one 64-channel chunk
        const int tid = threadIdx.x - 64;
        uint32_t a_it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int pt = tile / P.n_tiles_n;
            const int tx = pt % tiles_x, ty = (pt / tiles_x) % tiles_y, img = pt / (tiles_x * tiles_y);
            for (int c = 0; c < nchunks; ++c, ++a_it) {
                const uint32_t as = a_it % CV_A_BUFS, aph = (a_it / CV_A_BUFS) & 1u;
                mbar_wait_warp(&a_empty[as], aph ^ 1u);
                if ((P.dbg & 16) && a_it >= CV_A_BUFS) { mbar_arrive(&a_full[as]); continue; }
                conv_load_halo<HALO>(P, c, img, ty, tx, smem_u32(a_smem + as * CV_A_BUF_BYTES), tid);
                cp_async_mbar_arrive_noinc(&a_full[as]);   // arrives when this thread's copies have landed
            }
        }
    } else {
        // ================= epilogue: 8 warps; warp w reads TMEM lanes 32*(w%4).., warps 6-9 take the left 16x8 half
        // of the tile (sub 0), warps 10-13 the right one
        const int q = warp & 3;
        const int sub = (warp - 6) >> 2;
        uint32_t acc_it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++acc_it) {
            const int nt = tile % P.n_tiles_n, pt = tile / P.n_tiles_n;
            const int tx = pt % tiles_x, ty = (pt / tiles_x) % tiles_y, img = pt / (tiles_x * tiles_y);
            const uint32_t ab = acc_it & 1u;
            mbar_wait_warp(&acc_full[ab], (acc_it >> 1) & 1u);
            tc_fence_after_sync();
            const int y = ty * CV_TILE + 4 * q + (lane >> 3);
            const int x = tx * CV_TILE + 8 * sub + (lane & 7);
            const bool valid = (y < P.H) && (x < P.W) && !(P.dbg & 1);
            const uint32_t t0 = tmem_base + (static_cast<uint32_t>(32 * q) << 16) + ab * 256u + sub * 128u;
#pragma unroll 1
            for (int cc = 0; cc < ((P.dbg & 4) ? 0 : P.BN); cc += 32) {
                float v[32];
                tmem_ld32(t0 + cc, v);
                epi_store32<EK>(P.epi, has_bias ? bias_s : nullptr, v, img, y, x, nt * P.BN + cc, valid);
            }
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[ab]);
        }
    }

    // ---- teardown
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}

}  // namespace eb
