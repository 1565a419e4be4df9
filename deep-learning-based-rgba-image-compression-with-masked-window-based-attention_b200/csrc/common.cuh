// Blackwell (sm_100a) device primitives shared by the kernels of this library:
// mbarrier, bulk async copy (TMA engine, SASS UBLKCP), tcgen05 MMA / TMEM, UMMA descriptors.
// Hand-written inline PTX; nothing here comes from CUTLASS.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace b200 {

constexpr int kNumSMs = 148;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// immediate (non-suspending) probe of a phase
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

// generic-proxy smem writes -> visible to the async proxy (UMMA operand reads, bulk copies)
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------- bulk async copy (TMA engine, 1-D)
// global -> shared, completion signalled on an mbarrier via complete_tx.  bytes % 16 == 0.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---------------------------------------------------------------- TMEM
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {   // one full warp
    static_assert(kCols == 32 || kCols == 64 || kCols == 128 || kCols == 256 || kCols == 512, "pow2 >= 32");
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {     // same warp that allocated
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_wait_ld() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_wait_st() {
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// 32 lanes x 32 bit, N consecutive columns per thread: thread i of warp w reads TMEM lane 32*(w%4)+i.
__device__ __forceinline__ void tmem_ld_x8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}

// registers -> TMEM, same lane/column mapping as tmem_ld_x16
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}

__device__ __forceinline__ void tmem_ld_x4(uint32_t taddr, uint32_t (&r)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_st_x2(uint32_t taddr, uint32_t a, uint32_t b) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};" ::"r"(taddr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void tmem_st_x4(uint32_t taddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(a), "r"(b), "r"(c), "r"(d)
                 : "memory");
}
__device__ __forceinline__ void tmem_st_x8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
                 "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_x32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
        "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
        "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
        "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}

// ---------------------------------------------------------------- UMMA descriptors
// Shared-memory operand descriptor, K-major, SWIZZLE_128B canonical layout:
//   row r (M or N index), 16-byte chunk c (8 x 16-bit K elements) of a 64-element K block lives at
//   base + (r/8)*1024 + (r%8)*128 + ((c ^ (r%8)) * 16);   base must be 1024-byte aligned.
//   bits [0,14) start>>4 | [16,30) LBO>>4 (unused for swizzled K-major) | [32,46) SBO>>4 (=1024: next 8-row group)
//   | [46,48) version=1 | [61,64) layout type (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>(1) << 16;
    d |= static_cast<uint64_t>(1024 >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}
// byte offset of (row, k) for 16-bit elements inside one [rows x 64] K-major SW128 block
__device__ __host__ __forceinline__ uint32_t sw128_offset(uint32_t row, uint32_t k) {
    const uint32_t chunk = (k >> 3) ^ (row & 7u);
    return (row >> 3) * 1024u + (row & 7u) * 128u + chunk * 16u + (k & 7u) * 2u;
}

enum : uint32_t { kFmtF16 = 0, kFmtBF16 = 1, kFmtTF32 = 2 };
// kind::f16 / kind::tf32 instruction descriptor: fp32 accumulate, K-major A and B, dense.
__host__ __device__ constexpr uint32_t umma_idesc(uint32_t fmt_a, uint32_t fmt_b, uint32_t M, uint32_t N) {
    return (1u << 4) | (fmt_a << 7) | (fmt_b << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T, issued by ONE thread on behalf of the CTA.
__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Same with a lane mask: bit i of m[k] set = TMEM lane 32k + i of the accumulator is NOT written (tools/umma_probe.cu).
__device__ __forceinline__ void umma_f16_ss_lanes(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                  uint32_t accumulate, uint32_t m0, uint32_t m1, uint32_t m2, uint32_t m3) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(m0), "r"(m1), "r"(m2), "r"(m3)
        : "memory");
}
// Same with the A operand read from TMEM (16-bit elements packed two per 32-bit column: lane = row, column c holds
// k = 2c in the low and k = 2c + 1 in the high half; a k step of 16 = 8 columns).  Verified by tools/umma_ts_probe.cu.
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// A from TMEM with an output lane mask (see umma_f16_ss_lanes); verified by tools/umma_ts_probe.cu (mode `half`)
__device__ __forceinline__ void umma_f16_ts_lanes(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                                  uint32_t accumulate, uint32_t m0, uint32_t m1, uint32_t m2, uint32_t m3) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %6, %7, %8}, p;\n\t}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(m0), "r"(m1), "r"(m2), "r"(m3)
        : "memory");
}
// instruction-descriptor flag: the B operand is MN-major (stored [k][n], n contiguous; with SWIZZLE_128B the same
// physical layout as a K-major [rows = k][64] buffer).  Verified by tools/umma_ts_probe.cu.
constexpr uint32_t kUmmaBMajorMN = 1u << 16;
// All previously issued MMAs of this thread arrive (once) on `bar` when complete.
// Implies tcgen05.fence::before_thread_sync.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------- CTA pairs (tcgen05 cta_group::2) and clusters
// Verified on the hardware by tools/umma2_probe.cu: a cluster of 2 CTAs, each holding its own 128 A rows and HALF of
// the B rows, one M = 256 MMA issued by the leader, accumulator rows in each CTA's own TMEM, completion multicast to the
// mbarrier at the same shared-memory offset in both CTAs.
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {      // every thread of every CTA of the cluster
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of `local_smem_addr` (a shared::cta address) inside CTA `rank` of the cluster (shared::cluster window)
__device__ __forceinline__ uint32_t cluster_map_shared(uint32_t local_smem_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {   // arrive on another CTA's mbarrier
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem) {           // one warp in EACH CTA of the pair
    static_assert(kCols == 32 || kCols == 64 || kCols == 128 || kCols == 256 || kCols == 512, "pow2 >= 32");
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
// D[tmem of both CTAs] (+)= A[256 rows: 128 per CTA] * B[N rows: N/2 per CTA]^T; issued by ONE thread of the leader CTA.
// idesc: umma_idesc(fmt, fmt, 256, N).
__device__ __forceinline__ void umma_f16_ss_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                 uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// all previously issued pair MMAs of this thread arrive on the mbarrier at this offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t cta_mask = 3) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"(cta_mask)
                 : "memory");
}

// ---------------------------------------------------------------- TMA tensor copies (4-D tiled), verified by tools/tma_probe.cu
// `map` points at a CUtensorMap passed to the kernel as a __grid_constant__ parameter; coordinates innermost first.
__device__ __forceinline__ void tma_load_4d(void* dst_smem, const void* map, int c0, int c1, int c2, int c3, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2,%3,%4,%5}], [%6];" ::"r"(
            smem_u32(dst_smem)),
        "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tma_store_4d(const void* map, const void* src_smem, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2,%3,%4,%5}], [%1];" ::"l"(map),
                 "r"(smem_u32(src_smem)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
// global[box] += smem[box] (fp32), element-wise inside the L2; out-of-bound elements are skipped
__device__ __forceinline__ void tma_reduce_add_4d(const void* map, const void* src_smem, int c0, int c1, int c2, int c3) {
    asm volatile("cp.reduce.async.bulk.tensor.4d.global.shared::cta.add.tile.bulk_group [%0, {%2,%3,%4,%5}], [%1];" ::"l"(map),
                 "r"(smem_u32(src_smem)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int kPending>
__device__ __forceinline__ void bulk_wait_group_read() {   // smem sources of all but the last kPending groups consumed
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kPending) : "memory");
}
template <int kPending>
__device__ __forceinline__ void bulk_wait_group() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(kPending) : "memory");
}

// ---------------------------------------------------------------- small math / packing helpers
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ float bf16_round(float v) {   // nearest bf16 as fp32
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(0.f), "f"(v));
    return __uint_as_float(r << 16);
}

}  // namespace b200
