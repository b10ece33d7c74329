// common.cuh — sm_100a building blocks shared by every kernel of the EDVR hot path:
// mbarrier, tcgen05 (TMEM alloc / MMA / commit / ld), bulk-copy and proxy-fence wrappers,
// shared-memory matrix descriptors for the canonical *no-swizzle, K-major* UMMA layout.
//
// Layout convention used by all tensor-core kernels in this repo
// ---------------------------------------------------------------
// Operands live in shared memory as planes of 16-byte "K atoms":
//     elem(row r, k) -> plane (k / 8), row r, 8 halfs contiguous     (fp16 / bf16)
// i.e. byte address = base + (k/8) * LBO + (r/8) * SBO + (r%8) * 16 + (k%8) * 2.
// A "core matrix" (8 rows x 16 B) is therefore 128 contiguous bytes whenever rows are
// consecutive pixels / output channels, LBO is the plane pitch and SBO the pitch between
// 8-row groups.  That is the INTERLEAVE (no swizzle) canonical K-major layout
// ((8,n),2):((1,SBO),LBO) in 16-byte units.  Because rows are plain 16-byte slots,
// a 3x3 tap shift of an activation tile is just a different start address inside the same
// halo tile: one load of the halo serves all nine taps.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace eb {

// ---------------------------------------------------------------- error codes (C ABI)
enum : int {
    EB_OK = 0,
    EB_ERR_INVALID_SHAPE = -1,
    EB_ERR_UNSUPPORTED = -2,
    EB_ERR_LAUNCH = -3,
    EB_ERR_WORKSPACE = -4,
    EB_ERR_NULLPTR = -5,
    EB_ERR_ALIGNMENT = -6,
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
// Bounded wait: a protocol bug must become a trap (an error the host sees), never a hang.
// Inlined: a __noinline__ version (to shrink the code) added ~200 cycles per pipeline stage to the MMA issuer.
// Blocking try_wait (hardware sleep).  A non-blocking test_wait + __nanosleep back-off and warp-elected polling
// were both measured slower (wake-up latency; profiles/r01_conv_stats_*).
template <int SLEEP_NS = 32>
__device__ __forceinline__ void mbar_wait_t(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    long long t0 = 0;
    for (uint32_t spin = 0;; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
        if (done) break;
        if (SLEEP_NS > 0) __nanosleep(SLEEP_NS);
        if (spin == 64) t0 = clock64();
        if (spin > 64 && (spin & 1023u) == 0 && clock64() - t0 > 4000000000ll) __trap();
    }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) { mbar_wait_t<0>(bar, parity); }

// Wait with a suspend-time hint (nanoseconds, run-time value; 0 = the plain loop above).  Without a hint try_wait gives up
// after ~70 cycles and the loop around it re-issues ~8 instructions: nine waiting warps of the CTA-pair DCN kernel (issuers,
// producers, forwarder, epilogue) spent a quarter of the SM's issue slots spinning while the 16 gather warps were issue
// bound (profiles/r02_ncu_dcn_pair_v2: 60 % of all executed instructions were wait loops).  With a hint the thread sleeps in
// the SYNCS unit until the phase completes or the time is up.
__device__ __forceinline__ void mbar_wait_hint(uint64_t* bar, uint32_t parity, uint32_t hint_ns) {
    if (hint_ns == 0) { mbar_wait_t<0>(bar, parity); return; }
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    long long t0 = 0;
    for (uint32_t spin = 0;; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity), "r"(hint_ns)
            : "memory");
        if (done) break;
        if (spin == 64) t0 = clock64();
        if (spin > 64 && (spin & 1023u) == 0 && clock64() - t0 > 4000000000ll) __trap();
    }
}

// Same, observing arrivals made by the other CTA of the cluster (acquire at cluster scope).
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    long long t0 = 0;
    for (uint32_t spin = 0;; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
        if (done) break;
        if (spin == 64) t0 = clock64();
        if (spin > 64 && (spin & 1023u) == 0 && clock64() - t0 > 4000000000ll) __trap();
    }
}

// Whole-warp wait.  Every lane polls: electing one lane + __syncwarp (and try_wait suspend-time hints) measured
// 20-50 % SLOWER on B200 (profiles/r01_conv_stats_warp_elected.log) - the wake-up latency dominates.
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity) { mbar_wait(bar, parity); }

// ---------------------------------------------------------------- proxy / tcgen05 fences
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ---------------------------------------------------------------- TMEM allocation (one warp)
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(dst_smem)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
}

// ---------------------------------------------------------------- descriptors
// Shared-memory matrix descriptor (sm_100 "version 1"), no swizzle, K-major.
//   bits [0,14)  start address >> 4        bits [16,30) leading byte offset >> 4 (K pitch)
//   bits [32,46) stride byte offset >> 4   bits [46,48) version = 1
//   bits [61,64) layout type = 0 (SWIZZLE_NONE / interleave)
__device__ __forceinline__ uint64_t umma_desc_nosw(uint32_t saddr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFFu);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= 1ull << 46;
    return d;
}
// Instruction descriptor for kind::f16, fp32 accumulate, both operands K-major.
//   [4,6) c_format=1(F32) [7,10) a_format [10,13) b_format (0=F16, 1=BF16)
//   [17,23) N>>3   [24,29) M>>4
__host__ __device__ constexpr uint32_t umma_idesc_f16(uint32_t M, uint32_t N, uint32_t ab_fmt = 0) {
    return (1u << 4) | (ab_fmt << 7) | (ab_fmt << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T ; one thread issues for the whole CTA.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                         uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives once every MMA issued so far by this thread has completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                     smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------- CTA pairs (cta_group::2)
// Two CTAs of a cluster (same TPC) execute one M=256 MMA: rows [0,128) of A and D live in the even CTA, rows
// [128,256) in the odd one; B is split along N (first half in the even CTA).  Descriptors are interpreted at the
// same shared-memory offsets in both CTAs; only the even ("leader") CTA issues.
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t ncols) {   // one warp in EACH CTA
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// the mbarrier at this offset in every CTA of `cta_mask` receives one arrival when the MMAs issued so far are done
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"(cta_mask)
                 : "memory");
}
// arrive on the mbarrier at the same offset in CTA `target` of the cluster (release at cluster scope)
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t target) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(smem_u32(bar)), "r"(target)
        : "memory");
}
// Same signal WITHOUT a cluster-scope release (what CUTLASS' ClusterBarrier::arrive(cta_id) emits).  The .release.cluster
// form compiles to MEMBAR.ALL.GPU + ERRBAR + CGAERRBAR in front of the arrive (~0.3 us each, profiles/r02_ncu_dcn_pair_v1):
// fine once per tile, ruinous once per pipeline stage.  Use it when the arrival only tells the peer "go": the data it
// announces never crosses the CTA boundary through the generic proxy (shared memory read by the local tensor core after a
// local fence.proxy.async, or tensor memory whose reads were fenced with tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void mbar_arrive_remote_cta(uint64_t* bar, uint32_t target) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(smem_u32(bar)), "r"(target)
        : "memory");
}
// ---- lean issue path.  The MMA warp runs its loops with all 32 lanes converged and elects ONE lane per instruction:
// written like this the compiler keeps descriptors in uniform registers.  Issued from inside an `if (lane == 0)` region
// every MMA was wrapped in an election loop with 2-3 R2UR transfers (~15 dependent instructions, ~130 cycles per MMA
// for a 64-cycle MMA: the tensor pipe starved on issue, not on data; profiles/r01_one_conv_dbg.log).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// descriptor = {lo: start address >> 4 | LBO >> 4 << 16, hi: SBO >> 4 | version 1 << 14 | layout << 29}
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t saddr, uint32_t lbo_bytes) {
    return ((saddr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
__host__ __device__ constexpr uint32_t umma_desc_hi(uint32_t sbo_bytes) { return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14); }
template <int CG>
__device__ __forceinline__ void umma_f16_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                              uint32_t idesc, uint32_t accumulate) {
    if (CG == 2)
        asm volatile(
            "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
            "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
            "setp.ne.b32 p, %6, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}"
            ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
            : "memory");
    else
        asm volatile(
            "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
            "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
            "setp.ne.b32 p, %6, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
            ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
            : "memory");
}

// ---- TMA (tensor-map bulk copies), CTA-pair flavour: the copy lands in THIS CTA's shared memory, its bytes are
// counted on the mbarrier at the same offset in the EVEN CTA of the pair (the one that issues the MMAs).
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;     // clears the CTA-rank bit of a shared::cluster address
__device__ __forceinline__ void tma_load_5d_pair(void* dst_smem, const void* tmap, uint64_t* bar, int c0, int c1, int c2,
                                                 int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(smem_u32(dst_smem)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar) & kPeerBitMask),
          "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(void* dst_smem, const void* tmap, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst_smem)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
        : "memory");
}
// arrive + expect `bytes` on the mbarrier at the same offset in CTA `target` of the cluster
__device__ __forceinline__ void mbar_arrive_expect_tx_remote(uint64_t* bar, uint32_t bytes, uint32_t target) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.expect_tx.shared::cluster.b64 _, [ra], %2;\n\t}"
        ::"r"(smem_u32(bar)), "r"(target), "r"(bytes)
        : "memory");
}
// plain (single-CTA) tensor-map loads: the box lands in this CTA's shared memory, bytes counted on its own mbarrier
__device__ __forceinline__ void tma_load_3d(void* dst_smem, const void* tmap, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst_smem)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// shared -> global tile store (bulk async group of the issuing thread); out-of-range parts of the box are clipped
__device__ __forceinline__ void tma_store_4d(const void* tmap, const void* src_smem, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(src_smem)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}

// ---- programmatic dependent launch: a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may start
// while its predecessor in the stream is still running (once every CTA of the predecessor has triggered or exited); it must
// not touch memory the predecessor reads or writes before pdl_wait() returns (= predecessor complete and flushed).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Shared-memory matrix descriptor with a swizzled K-major layout (rows of 32/64/128 bytes, 8-row groups SBO apart):
// layout type 2 = 128 B, 4 = 64 B, 6 = 32 B swizzle.
__device__ __forceinline__ uint64_t umma_desc_sw(uint32_t saddr, uint32_t sbo_bytes, uint32_t layout_type) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFFu);
    d |= static_cast<uint64_t>(1u) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= 1ull << 46;
    d |= static_cast<uint64_t>(layout_type & 7u) << 61;
    return d;
}

// TMEM -> registers: this thread's lane (row), 32 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
          "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
          "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
          "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
          "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// ---------------------------------------------------------------- bulk async copy (global -> smem)
// 1-D, 16-byte aligned, size multiple of 16; completion counted in bytes on `bar`.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                         uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// same copy delivered to the same shared-memory offset of every CTA in `cta_mask` of the cluster; each destination CTA's
// mbarrier at the offset of `bar` receives the complete_tx (L2 is read once for the whole cluster)
__device__ __forceinline__ void bulk_g2s_multicast(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar,
                                                   uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::
            "r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "h"(cta_mask)
        : "memory");
}
// tcgen05.commit (cta_group::1) whose arrival is delivered to the mbarrier at this offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_multicast(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"(cta_mask)
                 : "memory");
}

// ---------------------------------------------------------------- small helpers
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
// 16-byte asynchronous global->shared copy (LDGSTS, L2-only); src_bytes == 0 writes zeros (image padding).
__device__ __forceinline__ void cp_async16_zfill(uint32_t saddr, const void* g, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(saddr), "l"(g), "r"(src_bytes) : "memory");
}
// The mbarrier receives one of its expected arrivals when all cp.async issued so far by this thread have landed.
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint64_t* bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32-byte read-only load (sm_100: LDG.256); p must be 32-byte aligned
__device__ __forceinline__ void ldg_nc_v8(const void* p, uint4& lo, uint4& hi) {
    asm volatile("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w), "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w)
                 : "l"(p));
}
__device__ __forceinline__ void sts_u32(uint32_t saddr, uint32_t v) {
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t saddr) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(saddr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_v4(uint32_t saddr, uint4 v) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y),
                 "r"(v.z), "r"(v.w)
                 : "memory");
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_bf2(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_h2(uint32_t u) {
    return __half22float2(*reinterpret_cast<__half2*>(&u));
}
__device__ __forceinline__ float sigmoidf_fast(float x) { return 1.0f / (1.0f + __expf(-x)); }

// activation codes shared by host and device
enum : int { ACT_NONE = 0, ACT_RELU = 1, ACT_LRELU = 2, ACT_SIGMOID = 4 };

__device__ __forceinline__ float apply_act(float v, int act) {
    if (act == ACT_RELU) return fmaxf(v, 0.0f);
    if (act == ACT_LRELU) return v > 0.0f ? v : 0.1f * v;
    if (act == ACT_SIGMOID) return sigmoidf_fast(v);
    return v;
}

// activation over a register tile with ONE dispatch (a per-element runtime switch compiles to a chain of
// uniform branches per element and made the epilogues branch-latency bound, profiles/r01_conv_stats_*.log)
template <int NV>
__device__ __forceinline__ void act_inplace(float (&v)[NV], int act) {
    if (act == ACT_RELU) {
#pragma unroll
        for (int j = 0; j < NV; ++j) v[j] = fmaxf(v[j], 0.0f);
    } else if (act == ACT_LRELU) {
#pragma unroll
        for (int j = 0; j < NV; ++j) v[j] = fmaxf(v[j], 0.1f * v[j]);     // == v > 0 ? v : 0.1 v
    } else if (act == ACT_SIGMOID) {
#pragma unroll
        for (int j = 0; j < NV; ++j) v[j] = sigmoidf_fast(v[j]);
    }
}

}  // namespace eb
