// Fused masked window attention forward in SPLIT PRECISION (fp32-faithful results on the tensor cores), sm_100a only.
// Reference semantics: layers/masked_win_attention.py:169-251 (block) and :96-131 (window attention), whose arithmetic
// is fp32 end to end.  A single fp16 pass per contraction misses the 1e-3 rel / 1e-4 abs contract on
// ~0.1 % of the outputs at random init and by far more on weights with large logits; tools/precision_study.py shows
// which operand roundings cost what.  Here EVERY operand of EVERY contraction (x, Wqkv, q, k, v, P, O, Wproj) is carried
// as fp16 hi + lo and contracted in three passes (hi*hi + lo*hi + hi*lo, fp32 accumulation in TMEM): ~2^-21 relative
// per product instead of 2^-11.
//
// One thread owns one token (= TMEM lane) from the QKV drain to the projection epilogue; only K and V go through
// shared memory (they are B operands), everything else stays in TMEM:
//
//   tile = 128 tokens = 2 kept 8x8 windows (rows 0-63 window slot 0, 64-127 slot 1), one head at a time:
//   QKV(h)   D_qkv[128 x 3d] = X_hi Wh_hi^T + X_lo Wh_hi^T + X_hi Wh_lo^T        (X_hi in shared memory, X_lo in TMEM)
//   drain    thread = token: q (+bias, pre-scaled by scale*log2e) -> fp16 hi / lo in TMEM (A operand of S);
//            k, v -> fp16 hi / lo rows in shared memory
//   S(h)     [128 x 64]: rows of window slot w against the 64 keys of slot w: two lane-masked MMAs per k step and pass
//   softmax  thread = (row, half of the keys): + relative-position bias (+ SW-MSA region mask), exp2, row sum;
//            P -> fp16 hi / lo written back over S in TMEM (A operand of P V)
//   PV(h)    O[128 x d] = P V_w  (V is the MN-major B operand [key][slot 0 d | slot 1 d]; again two lane-masked MMAs,
//            the second with its operand start advanced by d columns inside the swizzle atom)
//   norm     thread = row: O / rowsum -> fp16 hi / lo in TMEM over O (A operand of the projection)
//   proj(h)  D_out[128 x 192] += O_h Wproj_h^T, accumulated over the heads in TMEM
//   residual D_out is INITIALISED with x itself (X_hi I + X_lo I, 16-column identity MMAs, exact to 2^-22), so the
//            epilogue is a plain store of D_out + bias: no second read of x, no reduction, no pre-copy of the tensor.
//
// The issuer runs the heads as a software pipeline: slot G issues  P V(G) | S(G+1) | QKV(G+2) | proj(G)  so that the
// QKV and projection MMAs fill the tensor pipe while the softmax warps work on S(G+1); the tensor pipe executes in
// issue order, which is what makes the in-place reuse (P over S, the projection operand over O) safe without waits.
//
// Roles (24 warps, setmaxnreg): 0 MMA issuer | 1 weight feeder (two rings of bulk copies) | 2-3 TMA gather issuers
// (one per window slot, [16 ch][8][8] boxes of x) | 4-11 x converter + epilogue (fp32 boxes -> X_hi in shared memory,
// X_lo kept in registers until the previous tile's last QKV MMA has retired, then stored to TMEM; epilogue of the
// previous tile first) | 12-19 softmax (two warps per lane quarter) | 20-23 QKV drain + normalisation.
// Dropped windows are copied through by a separate small kernel (only the dropped ones).
#include <cstring>
#include <cuda.h>          // CUtensorMap (type only: the encoder is fetched through cudaGetDriverEntryPoint)
#include "mwa_lists.cuh"

// bring-up switches (tools/build_variants.py)
#ifndef MWA_SP_NO_TMA
#define MWA_SP_NO_TMA 0          // 1: every window through the LSU gather
#endif
#ifndef MWA_SP_EPI_NOSTORE
#define MWA_SP_EPI_NOSTORE 0     // 1: (debug) epilogue without its global stores
#endif

namespace b200 {
namespace {

constexpr int kSpWarps = 24;
constexpr int kSpThreads = kSpWarps * 32;
constexpr int kSpMma = 0, kSpFeed = 1, kSpTma0 = 2;
constexpr int kSpPe0 = 4, kSpNumPe = 8, kSpSm0 = 12, kSpNumSm = 8, kSpDr0 = 20;
// register pool of the CTA = 24 warps x 80 (launch bound); per SM sub-partition 56 + 2 x 88 + 2 x 80 + 88 = 480 = 6 x 80
constexpr int kSpRegsCtl = 56, kSpRegsPe = 88, kSpRegsSm = 80, kSpRegsDr = 88;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kNegMaskL2 = kNegMask * kLog2e;

template <int HEADS_>
struct SpCfg {
    static constexpr int C = 192, WS = 8, NTOK = 64, HEADS = HEADS_, D = C / HEADS;
    static_assert(D == 24 || D == 32, "head dim 24 / 32");
    static constexpr int KB = 3, KSTEPS = 12;
    // QKV weight ring element = (head, 64-channel K block, part): rows [q d][k d][v d] of the fp16 hi (part 0) or lo
    // (part 1) image, 128 B per row (K-major SW128), one bulk copy.  N of the QKV MMAs is 3d rounded up to a multiple
    // of 16: for d = 24 the 8 rows past the element are whatever follows in shared memory and only feed accumulator
    // columns 72-79, which nobody reads.
    static constexpr int NQ = (3 * D + 15) / 16 * 16;
    static constexpr uint32_t kWqElem = 3 * D * 128;
    static constexpr int kWqSlots = (D == 24) ? 4 : 3;
    static constexpr uint32_t kWpChunk = 96 * 128;
    static constexpr int TBL = 225;
    // TMEM columns: D_qkv | D_out | S (P hi / lo in place) | O (projection operand in place) | Q hi, lo | X_lo
    static constexpr uint32_t tDq = 0, tPj = 96, tS = 288, tO = 352, tOA = tO, tQ = 384, tXl = 416;
    static_assert(NQ <= 96, "TMEM budget");
    // shared memory map
    static constexpr uint32_t oXh = 0;                       // 2 x (KB x [128 x 64] fp16)
    static constexpr uint32_t oK = 2 * 49152;                // [128 keys] x 128 B: k hi (64 B) | k lo (64 B) of the head
    static constexpr uint32_t oVh = oK + 16384, oVl = oVh + 8192;   // [64 keys] x 128 B: [slot 0 d | slot 1 d]
    static constexpr uint32_t oWq = oVl + 8192;              // kWqSlots elements
    static constexpr uint32_t oWp = oWq + kWqSlots * kWqElem;    // 2 slots
    static constexpr uint32_t oStage = oWp + 2 * kWpChunk;   // 3 slots x 2 windows x 4 KB
    static constexpr uint32_t oI16 = oStage + 24576;
    static constexpr uint32_t oTbl = oI16 + 2048;
    static constexpr uint32_t oBq = (oTbl + HEADS * TBL * 4 + 15) / 16 * 16;
    static constexpr uint32_t oBpf = oBq + C * 4;
    static constexpr uint32_t oXch = oBpf + C * 4;            // fp32 row max [column half][128] | row sums [head parity][column half][128]
    static constexpr uint32_t oBars = oXch + 3072;
    static constexpr uint32_t oTmem = oBars + 64 * 8;
    static constexpr uint32_t oTotal = oTmem + 16;
    static_assert(oTotal <= 227 * 1024, "shared memory budget");
    static_assert(kWqElem % 1024 == 0 && oWq % 1024 == 0 && oWp % 1024 == 0 && oI16 % 1024 == 0, "operand alignment");
    // barriers
    static constexpr int bXhFull = 0, bXhEmpty = 2, bXlFull = 4, bXlEmpty = 5, bWqFull = 6, bWqEmpty = 10, bWpFull = 14,
                         bWpEmpty = 16, bDqFull = 18, bDqEmpty = 19, bQkReady = 20, bVReady = 21, bQkFree = 22, bVFree = 23,
                         bSFull = 24, bPReady = 25, bOFull = 26, bOAReady = 27, bPjFull = 28, bPjEmpty = 29,
                         bStFull = 30, bStEmpty = 36, bEnd = 42;
    static_assert(bEnd <= 64, "barrier slots");
};

// layout of the split-precision section of the parameter block (offsets from MwaParamLayout::img_sp)
template <class CF>
struct SpParams {
    static constexpr int64_t wq = 0;                                                   // [HEADS][KB][hi, lo] x kWqElem
    static constexpr int64_t wp = wq + int64_t(CF::HEADS) * CF::KB * 2 * CF::kWqElem;  // [HEADS][2] x kWpChunk
    static constexpr int64_t bq = wp + int64_t(CF::HEADS) * 2 * CF::kWpChunk;          // fp32 [C]  q bias * scale * log2e
    static constexpr int64_t bpf = bq + CF::C * 4;                                     // fp32 [C]  proj.bias + Wproj b_v
    static constexpr int64_t tbl = bpf + CF::C * 4;                                    // fp32 [HEADS][TBL] * log2e
    static constexpr int64_t i16 = tbl + (int64_t(CF::HEADS) * CF::TBL * 4 + 1023) / 1024 * 1024;
    static constexpr int64_t total = i16 + 2048;
};

__global__ void zero16_kernel(uint4* p, int64_t n16) {
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n16; i += int64_t(gridDim.x) * blockDim.x)
        p[i] = make_uint4(0, 0, 0, 0);
}

__device__ __forceinline__ uint16_t f16_bits(float v) { return __half_as_ushort(__float2half_rn(v)); }
__device__ __forceinline__ float f16_round(float v) { return __half2float(__float2half_rn(v)); }

template <class CF>
__global__ void mwa_sp_prepare_kernel(const float* __restrict__ qkv_w, const float* __restrict__ qkv_b,
                                      const float* __restrict__ proj_w, const float* __restrict__ proj_b,
                                      const float* __restrict__ table, float scale, uint8_t* __restrict__ out) {
    constexpr int C = CF::C, D = CF::D, H = CF::HEADS;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    const float qs = scale * kLog2e;
    for (int e = tid; e < H * CF::KB * 3 * D * 64; e += nth) {
        const int h = e / (CF::KB * 3 * D * 64), kb = (e / (3 * D * 64)) % CF::KB, n = (e / 64) % (3 * D), kk = e % 64;
        const int part = n / D, c = n % D;
        float w = qkv_w[int64_t(part * C + h * D + c) * C + kb * 64 + kk];
        if (part == 0) w *= qs;
        uint8_t* elem = out + SpParams<CF>::wq + int64_t((h * CF::KB + kb) * 2) * CF::kWqElem;
        const float hi = f16_round(w);
        *reinterpret_cast<uint16_t*>(elem + sw128_offset(n, kk)) = f16_bits(w);
        *reinterpret_cast<uint16_t*>(elem + CF::kWqElem + sw128_offset(n, kk)) = f16_bits(w - hi);
    }
    for (int e = tid; e < H * 2 * 96 * D; e += nth) {
        const int h = e / (2 * 96 * D), nh = (e / (96 * D)) % 2, n = (e / D) % 96, kk = e % D;
        const float w = proj_w[int64_t(nh * 96 + n) * C + h * D + kk];
        uint8_t* chunk = out + SpParams<CF>::wp + int64_t(h * 2 + nh) * CF::kWpChunk;
        const float hi = f16_round(w);
        *reinterpret_cast<uint16_t*>(chunk + sw128_offset(n, kk)) = f16_bits(w);
        *reinterpret_cast<uint16_t*>(chunk + sw128_offset(n, 32 + kk)) = f16_bits(w - hi);
    }
    for (int c = tid; c < C; c += nth) {
        reinterpret_cast<float*>(out + SpParams<CF>::bq)[c] = qkv_b ? qkv_b[c] * qs : 0.f;
        float v = proj_b[c];
        if (qkv_b != nullptr)
            for (int k = 0; k < C; ++k) v = fmaf(proj_w[int64_t(c) * C + k], qkv_b[2 * C + k], v);
        reinterpret_cast<float*>(out + SpParams<CF>::bpf)[c] = v;
    }
    for (int e = tid; e < H * CF::TBL; e += nth)
        reinterpret_cast<float*>(out + SpParams<CF>::tbl)[e] = table[(e % CF::TBL) * H + e / CF::TBL] * kLog2e;
    for (int n = tid; n < 16; n += nth)
        *reinterpret_cast<uint16_t*>(out + SpParams<CF>::i16 + sw128_offset(n, n)) = f16_bits(1.0f);
}

// ------------------------------------------------------------------------------------------------ small helpers
template <int N>
__device__ __forceinline__ void sp_reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void sp_reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
__device__ __forceinline__ void sp_st_shared_f32(uint32_t addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void sp_named_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ float sp_ld_shared_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
// fp16 hi / lo split of two values: hi = rn(v), lo = rn(v - hi), packed (first value in the low half)
__device__ __forceinline__ void split_f16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(a, b);
    const float2 hf = __half22float2(h);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = pack_f16x2(a - hf.x, b - hf.y);
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ float ex2(float v) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float max3(float a, float b, float c) {
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

template <class CF, bool kTiming>
__global__ void __launch_bounds__(kSpThreads, 1)
mwa_sp_kernel(const float* __restrict__ x, float* __restrict__ out, const uint8_t* __restrict__ sp,
              const int32_t* __restrict__ list, const int32_t* __restrict__ count_p, Geom geo,
              unsigned long long* __restrict__ timing, const __grid_constant__ CUtensorMap x_map) {
    constexpr int C = CF::C, WS = CF::WS, D = CF::D, H = CF::HEADS;
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t sb = smem_u32(smem);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + CF::oBars);
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + CF::oTmem);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    // ---- one-time setup
    if (tid == 0) {
        if (sb & 1023u) __trap();
        for (int i = 0; i < 2; ++i) {
            mbar_init(bars + CF::bXhFull + i, kSpNumPe * 32);
            mbar_init(bars + CF::bXhEmpty + i, 1);
            mbar_init(bars + CF::bWpFull + i, 1);
            mbar_init(bars + CF::bWpEmpty + i, 1);
        }
        for (int i = 0; i < CF::kWqSlots; ++i) {
            mbar_init(bars + CF::bWqFull + i, 1);
            mbar_init(bars + CF::bWqEmpty + i, 1);
        }
        mbar_init(bars + CF::bXlFull, kSpNumPe * 32);
        mbar_init(bars + CF::bXlEmpty, 1);
        mbar_init(bars + CF::bDqFull, 1);
        mbar_init(bars + CF::bDqEmpty, 128);
        mbar_init(bars + CF::bQkReady, 128);
        mbar_init(bars + CF::bVReady, 128);
        mbar_init(bars + CF::bQkFree, 1);
        mbar_init(bars + CF::bVFree, 1);
        mbar_init(bars + CF::bSFull, 1);
        mbar_init(bars + CF::bPReady, kSpNumSm * 32);
        mbar_init(bars + CF::bOFull, 1);
        mbar_init(bars + CF::bOAReady, 128);
        mbar_init(bars + CF::bPjFull, 1);
        mbar_init(bars + CF::bPjEmpty, kSpNumPe * 32);
        for (int i = 0; i < 6; ++i) {
            mbar_init(bars + CF::bStFull + i, 1);
            mbar_init(bars + CF::bStEmpty + i, 128);
        }
        fence_mbar_init();
    }
    if (warp == kSpFeed) tmem_alloc<512>(tmem_ptr);
    {
        const float* gt = reinterpret_cast<const float*>(sp + SpParams<CF>::tbl);
        float* st = reinterpret_cast<float*>(smem + CF::oTbl);
        for (int i = tid; i < H * CF::TBL; i += kSpThreads) st[i] = gt[i];
        const float* gb = reinterpret_cast<const float*>(sp + SpParams<CF>::bq);       // bq and bpf are adjacent
        float* sbq = reinterpret_cast<float*>(smem + CF::oBq);
        for (int i = tid; i < 2 * C; i += kSpThreads) sbq[i] = gb[i];
        const uint4* gi = reinterpret_cast<const uint4*>(sp + SpParams<CF>::i16);
        for (int i = tid; i < 2048 / 16; i += kSpThreads) reinterpret_cast<uint4*>(smem + CF::oI16)[i] = gi[i];
        // K and V rows incl. their pad chunks: must read as zeros (finite) wherever nothing is written
        for (int i = tid; i < (CF::oWq - CF::oK) / 16; i += kSpThreads)
            reinterpret_cast<uint4*>(smem + CF::oK)[i] = make_uint4(0, 0, 0, 0);
    }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tm = *tmem_ptr;

    const int count = *count_p;
    const int num_tiles = (count + 1) / 2;
    const int64_t hw = int64_t(geo.H) * geo.W;
    auto tile_of = [&](int it) -> int { return it * int(gridDim.x) + int((blockIdx.x + unsigned(it)) % gridDim.x); };
    int my_tiles;
    {
        const int full = num_tiles / int(gridDim.x), rem = num_tiles - full * int(gridDim.x);
        my_tiles = full + ((int((blockIdx.x + unsigned(full)) % gridDim.x) < rem) ? 1 : 0);
    }
    const int total = my_tiles * H;                       // heads this CTA processes (global head index G = it * H + h)
    const long long t_cta0 = (kTiming && timing != nullptr) ? clock64() : 0;
    // development aid (kTiming instantiation only): event trace of CTA 0, first lane of the first warp of each role:
    // timing[1024 + role * 1024 + i] = stage << 48 | cycles since kernel start at the END of the stage (buffer: 8192 u64)
    const bool do_time = kTiming && timing != nullptr && blockIdx.x == 0 && lane == 0 &&
                         (warp == kSpMma || warp == kSpPe0 || warp == kSpSm0 || warp == kSpDr0);
    int n_ev = 0;
    auto tick = [&](int slot) {
        if constexpr (kTiming) {
            if (do_time && n_ev < 1024)
                timing[1024 + (slot >> 3) * 1024 + n_ev++] =
                    (static_cast<unsigned long long>(slot) << 48) | static_cast<unsigned long long>(clock64() - t_cta0);
        }
    };

    if (warp < 4) {
        // =========================================================================================== control warps
        sp_reg_dec<kSpRegsCtl>();
        if (warp == kSpMma && elect_one()) {
            // One elected thread of a CONVERGED warp (not `lane == 0`: a divergent branch makes every tcgen05.mma cost ~45
            // cycles of issue, tools/umma_rate_probe.cu) issues every MMA of the CTA.  Measured cost per MMA (M = 128,
            // K = 16): A from shared memory max(N/2, 32 + N/4) cycles, A from TMEM N/2.
            constexpr uint32_t id_q = umma_idesc(kFmtF16, kFmtF16, 128, CF::NQ), id_s = umma_idesc(kFmtF16, kFmtF16, 128, 64);
            constexpr uint32_t id_o = umma_idesc(kFmtF16, kFmtF16, 128, 32) | kUmmaBMajorMN;
            constexpr uint32_t id_p = umma_idesc(kFmtF16, kFmtF16, 128, 96), id_r = umma_idesc(kFmtF16, kFmtF16, 128, 16);
            const uint64_t d_x = umma_desc_k_sw128(sb + CF::oXh), d_wq = umma_desc_k_sw128(sb + CF::oWq),
                           d_wp = umma_desc_k_sw128(sb + CF::oWp), d_k = umma_desc_k_sw128(sb + CF::oK),
                           d_vh = umma_desc_k_sw128(sb + CF::oVh), d_vl = umma_desc_k_sw128(sb + CF::oVl),
                           d_i = umma_desc_k_sw128(sb + CF::oI16);
            uint32_t nq = 0, np = 0;                       // weight ring elements consumed from the two rings
            int next_q = 0;                                // next head whose QKV MMAs are to be issued
            // QKV(q) in three K blocks (so that other MMAs can be issued in between: the weight ring holds two K blocks and
            // refills in ~1 k cycles, a head's six elements back to back would outrun it)
            auto qkv_block = [&](int q, int kb) {
                const int it = q / H, h = q - it * H, xb = it & 1;
                if (kb == 0) {
                    if (h == 0) {
                        mbar_wait(bars + CF::bXhFull + xb, (it >> 1) & 1);
                        mbar_wait(bars + CF::bXlFull, it & 1);
                    }
                    if (q > 0) mbar_wait(bars + CF::bDqEmpty, (q - 1) & 1);
                    tc_fence_after_sync();
                }
                const uint64_t a0 = d_x + ((xb * 49152 + kb * 16384) >> 4);
                uint32_t slot = nq % CF::kWqSlots;
                mbar_wait(bars + CF::bWqFull + slot, (nq / CF::kWqSlots) & 1);      // W hi of the K block
                tc_fence_after_sync();
                uint64_t b0 = d_wq + ((slot * CF::kWqElem) >> 4);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    umma_f16_ss(tm + CF::tDq, a0 + ks * 2, b0 + ks * 2, id_q, (kb | ks) != 0);
                    umma_f16_ts(tm + CF::tDq, tm + CF::tXl + (kb * 4 + ks) * 8, b0 + ks * 2, id_q, 1);
                }
                umma_commit(bars + CF::bWqEmpty + slot);
                ++nq;
                slot = nq % CF::kWqSlots;
                mbar_wait(bars + CF::bWqFull + slot, (nq / CF::kWqSlots) & 1);      // W lo
                tc_fence_after_sync();
                b0 = d_wq + ((slot * CF::kWqElem) >> 4);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) umma_f16_ss(tm + CF::tDq, a0 + ks * 2, b0 + ks * 2, id_q, 1);
                umma_commit(bars + CF::bWqEmpty + slot);
                ++nq;
                if (kb == CF::KB - 1) {
                    umma_commit(bars + CF::bDqFull);
                    if (h == H - 1) {
                        umma_commit(bars + CF::bXhEmpty + xb);
                        umma_commit(bars + CF::bXlEmpty);
                    }
                }
            };
            auto issue_qkv = [&](int q) {
#pragma unroll
                for (int kb = 0; kb < CF::KB; ++kb) qkv_block(q, kb);
            };
            // S(G): rows 0-63 (window slot 0) against the keys of slot 0, rows 64-127 against those of slot 1: two MMAs per
            // k step with the other half of the output lanes disabled; passes q_hi k_hi + q_lo k_hi + q_hi k_lo
            auto issue_s = [&](int G) {
                mbar_wait(bars + CF::bQkReady, G & 1);
                tc_fence_after_sync();
#pragma unroll
                for (int pass = 0; pass < 3; ++pass) {
                    const uint32_t a = tm + CF::tQ + (pass == 1 ? 16 : 0);
                    const uint64_t b = d_k + (pass == 2 ? 4 : 0);
#pragma unroll
                    for (int ks = 0; ks < 2; ++ks) {
                        const uint32_t acc = (pass | ks) != 0;
                        umma_f16_ts_lanes(tm + CF::tS, a + ks * 8, b + ks * 2, id_s, acc, 0u, 0u, ~0u, ~0u);
                        umma_f16_ts_lanes(tm + CF::tS, a + ks * 8, b + 512 + ks * 2, id_s, acc, ~0u, ~0u, 0u, 0u);
                    }
                }
                umma_commit(bars + CF::bSFull);
                umma_commit(bars + CF::bQkFree);
            };
            // O(G) = P V: 16 keys per k step (= 2048 bytes of the [key][128 B] buffers), a row's own window is one d-wide
            // part of the V rows; N = 32 (>= d: columns d .. 31 of O receive finite junk that nobody reads)
            auto issue_pv = [&](int G) {
                mbar_wait(bars + CF::bVReady, G & 1);
                mbar_wait(bars + CF::bPReady, G & 1);
                tc_fence_after_sync();
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
                    for (int pass = 0; pass < 3; ++pass) {
                        const uint32_t a = tm + CF::tS + (pass == 1 ? 32 : 0) + ks * 8;
                        const uint64_t b = (pass == 2 ? d_vl : d_vh) + ks * 128;
                        const uint32_t acc = (pass | ks) != 0;
                        umma_f16_ts_lanes(tm + CF::tO, a, b, id_o, acc, 0u, 0u, ~0u, ~0u);
                        umma_f16_ts_lanes(tm + CF::tO, a, b + ((D * 2) >> 4), id_o, acc, ~0u, ~0u, 0u, 0u);
                    }
                }
                umma_commit(bars + CF::bOFull);
                umma_commit(bars + CF::bVFree);
            };
            auto proj_half = [&](int G, int nh) {
                const int it = G / H, h = G - it * H, xb = it & 1;
                if (nh == 0) {
                    mbar_wait(bars + CF::bOAReady, G & 1);
                    if (h == 0) {
                        // the accumulator starts as the residual x itself: D[:, 16j .. 16j+15] = X_hi(j) I + X_lo(j) I
                        if (it > 0) mbar_wait(bars + CF::bPjEmpty, (it - 1) & 1);
                        tc_fence_after_sync();
#pragma unroll
                        for (int ks = 0; ks < CF::KSTEPS; ++ks) {
                            umma_f16_ss(tm + CF::tPj + ks * 16, d_x + ((xb * 49152 + (ks >> 2) * 16384) >> 4) + (ks & 3) * 2, d_i, id_r, 0);
                            umma_f16_ts(tm + CF::tPj + ks * 16, tm + CF::tXl + ks * 8, d_i, id_r, 1);
                        }
                    }
                    tc_fence_after_sync();
                }
                const uint32_t slot = np & 1;
                mbar_wait(bars + CF::bWpFull + slot, (np >> 1) & 1);
                tc_fence_after_sync();
                const uint64_t b0 = d_wp + ((slot * CF::kWpChunk) >> 4);
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    umma_f16_ts(tm + CF::tPj + nh * 96, tm + CF::tOA + ks * 8, b0 + ks * 2, id_p, 1);
                    umma_f16_ts(tm + CF::tPj + nh * 96, tm + CF::tOA + 16 + ks * 8, b0 + ks * 2, id_p, 1);
                    umma_f16_ts(tm + CF::tPj + nh * 96, tm + CF::tOA + ks * 8, b0 + 4 + ks * 2, id_p, 1);
                }
                umma_commit(bars + CF::bWpEmpty + slot);
                ++np;
                if (nh == 1 && h == H - 1) umma_commit(bars + CF::bPjFull);
            };
            if (total > 0) {
                issue_qkv(next_q++);
                issue_s(0);
                if (next_q < total) issue_qkv(next_q++);
            }
            for (int G = 0; G < total; ++G) {
                issue_pv(G);
                tick(0);                                                         // 0: wait P, V + P V issue
                if (G + 1 < total) issue_s(G + 1);           // right behind P V(G): overwrites P(G) in issue order
                tick(1);                                                         // 1: wait Q, K + S issue
                // QKV(G + 2) and proj(G) fill the tensor pipe during softmax(G + 1), interleaved K block by K block
                const bool has_q = next_q < total;
                const int q = next_q;
                if (has_q) qkv_block(q, 0);
                if (has_q) qkv_block(q, 1);
                proj_half(G, 0);                             // its operand (O(G) normalised) is ~1 k cycles behind P V(G)
                if (has_q) {
                    qkv_block(q, 2);
                    ++next_q;
                }
                proj_half(G, 1);
                tick(2);                                                         // 2: QKV(G + 2) + proj(G) issue incl. their waits
            }
        } else if (warp == kSpFeed && elect_one()) {
            // weight feeder: two rings of bulk copies, each in exactly the order the issuer consumes it
            const uint8_t* gq = sp + SpParams<CF>::wq;
            const uint8_t* gp = sp + SpParams<CF>::wp;
            const uint32_t nQ = uint32_t(total) * CF::KB * 2, nP = uint32_t(total) * 2;
            uint32_t iq = 0, ip = 0;
            while (iq < nQ || ip < nP) {
                if (iq < nQ) {
                    const uint32_t slot = iq % CF::kWqSlots;
                    if (iq < uint32_t(CF::kWqSlots) || mbar_test_wait(bars + CF::bWqEmpty + slot, ((iq / CF::kWqSlots) - 1) & 1)) {
                        const uint32_t h = (iq / (CF::KB * 2)) % H, e = iq % (CF::KB * 2);      // e = kb * 2 + part
                        mbar_arrive_expect_tx(bars + CF::bWqFull + slot, CF::kWqElem);
                        bulk_g2s(smem + CF::oWq + slot * CF::kWqElem, gq + int64_t(h * CF::KB * 2 + e) * CF::kWqElem,
                                 CF::kWqElem, bars + CF::bWqFull + slot);
                        ++iq;
                    }
                }
                if (ip < nP) {
                    const uint32_t slot = ip & 1;
                    if (ip < 2 || mbar_test_wait(bars + CF::bWpEmpty + slot, ((ip >> 1) - 1) & 1)) {
                        const uint32_t h = (ip >> 1) % H, nh = ip & 1;
                        mbar_arrive_expect_tx(bars + CF::bWpFull + slot, CF::kWpChunk);
                        bulk_g2s(smem + CF::oWp + slot * CF::kWpChunk, gp + int64_t(h * 2 + nh) * CF::kWpChunk, CF::kWpChunk,
                                 bars + CF::bWpFull + slot);
                        ++ip;
                    }
                }
            }
        } else if (warp >= kSpTma0) {
            // TMA gather issuer of window slot w: 12 boxes [16 ch][8][8] per window, channel halves interleaved in the
            // order the converter warps consume them; windows that wrap round the image border are left to the LSU path
            const int w = warp - kSpTma0;
            uint32_t n = 0;
            for (int i = 0; i < my_tiles; ++i) {
                const int lidx = tile_of(i) * 2 + w;
                if (lidx >= count) continue;
                int b_, wy_, wx_;
                window_coords(geo, list[lidx], b_, wy_, wx_);
                const int x0 = wx_ * WS + geo.shift, y0 = wy_ * WS + geo.shift;
                if (MWA_SP_NO_TMA || x0 + WS > geo.W || y0 + WS > geo.H) continue;
                for (int j = 0; j < 12; ++j, ++n) {
                    const int k = (j & 1) * 6 + (j >> 1);
                    const uint32_t slot = n % 3;
                    if (n >= 3) mbar_wait(bars + CF::bStEmpty + w * 3 + slot, ((n / 3) - 1) & 1);
                    if (lane == 0) {
                        mbar_arrive_expect_tx(bars + CF::bStFull + w * 3 + slot, 4096);
                        tma_load_4d(smem + CF::oStage + (slot * 2 + w) * 4096, &x_map, x0, y0, k * 16, b_,
                                    bars + CF::bStFull + w * 3 + slot);
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp < kSpSm0) {
        // =========================================================================================== x converter + epilogue
        sp_reg_inc<kSpRegsPe>();
        const int pw = warp - kSpPe0, q = pw & 3, half = pw >> 2;
        const int r = q * 32 + lane, wslot = r >> 6, tok = r & 63;
        const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
        const float* s_bpf = reinterpret_cast<const float*>(smem + CF::oBpf);
        uint32_t lo[6][8];                                   // fp16 lo parts of this thread's 96 channels of the NEXT tile
        uint32_t stage_n = 0;                                // boxes of this thread's window slot consumed so far
        // per-tile window info of this thread's token
        struct Win {
            bool valid, staged;
            int64_t base;                                    // NCHW element offset of (b, c = 0, py, px)
        };
        auto win_of = [&](int tile) -> Win {
            Win wi;
            const int lidx = tile * 2 + wslot;
            wi.valid = lidx < count;
            int b, wy, wx, py, px;
            window_coords(geo, list[wi.valid ? lidx : (count - 1)], b, wy, wx);
            wi.staged = !MWA_SP_NO_TMA && wi.valid && (wx * WS + geo.shift + WS <= geo.W) && (wy * WS + geo.shift + WS <= geo.H);
            token_pixel<WS>(geo, wy, wx, tok, py, px);
            wi.base = int64_t(b) * C * hw + int64_t(py) * geo.W + px;
            return wi;
        };
        // box jj (0..11) of the window's stream: channels k*16 .. k*16+15 with k = (jj & 1) * 6 + (jj >> 1); this thread
        // converts the boxes of its own half.  EVERY thread of the window observes every box (a parity wait may lag an
        // mbarrier by one phase only).
        auto gather_box = [&](const Win& wi, int jj, int xb) {
            float v[16];
            uint64_t* release = nullptr;                     // staging slot to hand back once its values have been consumed
            if (wi.staged) {
                const uint32_t nb = stage_n + jj, slot = nb % 3;
                mbar_wait(bars + CF::bStFull + wslot * 3 + slot, (nb / 3) & 1);
                if ((jj & 1) != half) {
                    mbar_arrive(bars + CF::bStEmpty + wslot * 3 + slot);
                    return;
                }
                const uint32_t base = sb + CF::oStage + (slot * 2 + wslot) * 4096 + tok * 4;
#pragma unroll
                for (int c = 0; c < 16; ++c) v[c] = sp_ld_shared_f32(base + c * 256);
                release = bars + CF::bStEmpty + wslot * 3 + slot;
            } else {
                if ((jj & 1) != half) return;
                const float* p = x + wi.base + int64_t((half * 6 + (jj >> 1)) * 16) * hw;
#pragma unroll
                for (int c = 0; c < 16; ++c) v[c] = wi.valid ? __ldg(p + c * hw) : 0.f;
            }
            const int i = jj >> 1, k = half * 6 + i;
            uint32_t hi[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) split_f16x2(v[2 * j], v[2 * j + 1], hi[j], lo[i][j]);
#pragma unroll
            for (int c2 = 0; c2 < 2; ++c2) {
                const int ci = 2 * k + c2;                   // 8-channel chunk index 0..23
                const uint32_t addr = sb + CF::oXh + xb * 49152 + (ci >> 3) * 16384 + (r >> 3) * 1024 + (r & 7) * 128 +
                                      (((ci & 7) ^ (r & 7)) << 4);
                st_shared_v4(addr, hi[4 * c2], hi[4 * c2 + 1], hi[4 * c2 + 2], hi[4 * c2 + 3]);
            }
            // The slot is released only AFTER the loaded values have been used: an mbarrier arrive does not wait for
            // ld.shared instructions still queued in the LSU (behind the epilogue's global stores they can be hundreds of
            // cycles late), and the TMA would overwrite the box under them.  Seen on the hardware as stale tail channels.
            if (release != nullptr) mbar_arrive(release);
        };
        auto publish_lo = [&](int it_next) {                 // X_lo of tile it_next -> TMEM (columns = channel pairs)
#pragma unroll
            for (int i = 0; i < 6; ++i) tmem_st_x8(tm + CF::tXl + lane_addr + (half * 6 + i) * 8, lo[i]);
            tmem_wait_st();
            tc_fence_before_sync();
            mbar_arrive(bars + CF::bXlFull);
            (void)it_next;
        };
        if (my_tiles > 0) {
            const Win w0 = win_of(tile_of(0));
#pragma unroll
            for (int jj = 0; jj < 12; ++jj) gather_box(w0, jj, 0);
            if (w0.staged) stage_n += 12;
            fence_proxy_async_smem();
            mbar_arrive(bars + CF::bXhFull + 0);
            publish_lo(0);
        }
        // iteration `it` runs while tile `it` is computed: epilogue of tile it - 1, then the conversion of tile it + 1.
        // The issuer needs the projection accumulator back one head period after the tile's last projection (for the
        // residual MMAs of the next tile), so the epilogue hands it back as early as it can: the first 48 of a thread's
        // 96 columns go load -> store in steps of 8, the other 48 are read into registers in one go, the accumulator is
        // released, and only then are they stored.  (Interleaving the epilogue with the next conversion, as an earlier
        // version did, held the accumulator for ~16 k cycles and stalled the issuer at every tile boundary.)
        for (int it = 0; it <= my_tiles; ++it) {
            const bool do_epi = it >= 1, do_gather = it + 1 < my_tiles;
            if (!do_epi && !do_gather) continue;
            const int xb = (it + 1) & 1;
            if (do_epi) {
                const Win wp = win_of(tile_of(it - 1));
                float* orow = out + wp.base + int64_t(half * 96) * hw;
                const float* bp = s_bpf + half * 96;
                const bool store = wp.valid && !MWA_SP_EPI_NOSTORE;
                tick(8);                                                         // 8: tile set-up
                mbar_wait(bars + CF::bPjFull, (it - 1) & 1);
                tc_fence_after_sync();
                tick(9);                                                         // 9: wait projection complete
#pragma unroll
                for (int st = 0; st < 6; ++st) {
                    uint32_t acc[8];
                    tmem_ld_x8(tm + CF::tPj + lane_addr + half * 96 + st * 8, acc);
                    tmem_wait_ld();
                    if (store) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) orow[int64_t(st * 8 + j) * hw] = __uint_as_float(acc[j]) + bp[st * 8 + j];
                    }
                }
                uint32_t rest[6][8];
#pragma unroll
                for (int st = 0; st < 6; ++st) tmem_ld_x8(tm + CF::tPj + lane_addr + half * 96 + 48 + st * 8, rest[st]);
                tmem_wait_ld();
                tc_fence_before_sync();
                mbar_arrive(bars + CF::bPjEmpty);            // every column has been read: the accumulator goes back
                tick(13);                                                        // 13: (marker) accumulator released
                if (store) {
#pragma unroll
                    for (int st = 0; st < 6; ++st)
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            orow[int64_t(48 + st * 8 + j) * hw] = __uint_as_float(rest[st][j]) + bp[48 + st * 8 + j];
                }
            }
            if (do_gather) {
                const Win wn = win_of(tile_of(it + 1));
                if (it >= 1) mbar_wait(bars + CF::bXhEmpty + xb, ((it - 1) >> 1) & 1);
#pragma unroll
                for (int jj = 0; jj < 12; ++jj) gather_box(wn, jj, xb);
                if (wn.staged) stage_n += 12;
            }
            tick(10);                                                            // 10: epilogue stores + conversion
            if (do_gather) {
                fence_proxy_async_smem();
                mbar_arrive(bars + CF::bXhFull + xb);
                mbar_wait(bars + CF::bXlEmpty, it & 1);      // the correction MMAs of tile `it` have read X_lo
                tc_fence_after_sync();
                tick(11);                                                        // 11: wait X_lo free
                publish_lo(it + 1);
                tick(12);                                                        // 12: X_lo -> TMEM
            }
        }
    } else if (warp < kSpDr0) {
        // =========================================================================================== softmax
        // Two warps per 32-row lane quarter (both on the same SM sub-partition, as the TMEM lane rule demands): each takes
        // 32 of the row's 64 logits; the row max goes through shared memory and a 64-thread named barrier, the two partial
        // row sums are left in shared memory for the thread that normalises O (per head parity: it reads them one head later).
        sp_reg_inc<kSpRegsSm>();
        const int sw = warp - kSpSm0, q = sw & 3, ch = sw >> 2;
        const int r = q * 32 + lane, wslot = r >> 6, tok = r & 63;
        const int yi = tok >> 3, xi = tok & 7;
        const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
        // this lane's entry of the relative-position table for key 32 * ch (keys run down the table: - (yj * 15 + xj))
        const uint32_t tbl0 = sb + CF::oTbl + 4 * ((yi + WS - 1 - 4 * ch) * (2 * WS - 1) + xi + WS - 1);
        const uint32_t xmax_me = sb + CF::oXch + 4 * (ch * 128 + r), xmax_other = sb + CF::oXch + 4 * ((ch ^ 1) * 128 + r);
        const uint32_t xsum_me = sb + CF::oXch + 1024 + 4 * (ch * 128 + r);
        for (int it = 0; it < my_tiles; ++it) {
            // SW-MSA region mask bits of this row's 32 keys (:194-216); zero unless the window touches the wrapped border
            uint32_t mb = 0;
            bool has_mask = false;
            if (geo.shift > 0) {
                const int lidx = tile_of(it) * 2 + wslot;
                int b_, wy, wx;
                window_coords(geo, list[lidx < count ? lidx : count - 1], b_, wy, wx);
                has_mask = (wy == geo.nwy - 1) || (wx == geo.nwx - 1);
                if (has_mask) {
                    const int ys0 = wy * WS, xs0 = wx * WS;
                    const int by = (ys0 + yi >= geo.H - WS) + (ys0 + yi >= geo.H - geo.shift);
                    const int bx = (xs0 + xi >= geo.W - WS) + (xs0 + xi >= geo.W - geo.shift);
                    uint32_t dy = 0, dx = 0;
#pragma unroll
                    for (int j = 0; j < WS; ++j) {
                        dy |= uint32_t(((ys0 + j >= geo.H - WS) + (ys0 + j >= geo.H - geo.shift)) != by) << j;
                        dx |= uint32_t(((xs0 + j >= geo.W - WS) + (xs0 + j >= geo.W - geo.shift)) != bx) << j;
                    }
                    dy >>= 4 * ch;
#pragma unroll
                    for (int j = 0; j < 32; ++j) mb |= (((dy >> (j >> 3)) | (dx >> (j & 7))) & 1u) << j;
                }
            }
            for (int h = 0; h < H; ++h) {
                const int G = it * H + h;
                mbar_wait(bars + CF::bSFull, G & 1);
                tc_fence_after_sync();
                tick(16);                                                        // 16: wait S
                float s[32];
                {
                    uint32_t raw[32];
                    tmem_ld_x32(tm + CF::tS + lane_addr + ch * 32, raw);
                    tmem_wait_ld();
#pragma unroll
                    for (int j = 0; j < 32; ++j) s[j] = __uint_as_float(raw[j]);
                }
                // relative-position bias (layers/masked_win_attention.py:109-112), table pre-multiplied by log2(e)
                const uint32_t tb = tbl0 + h * (CF::TBL * 4);
#pragma unroll
                for (int j = 0; j < 32; ++j) s[j] += sp_ld_shared_f32(tb - 4 * ((j >> 3) * (2 * WS - 1) + (j & 7)));
                if (has_mask) {
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if ((mb >> j) & 1u) s[j] += kNegMaskL2;
                }
                float m = s[0];
#pragma unroll
                for (int j = 1; j < 31; j += 2) m = max3(m, s[j], s[j + 1]);
                m = fmaxf(m, s[31]);
                sp_st_shared_f32(xmax_me, m);
                sp_named_sync(1 + q, 64);
                m = fmaxf(m, sp_ld_shared_f32(xmax_other));
                float sum = 0.f;
                uint32_t ph[16], pl[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float p0 = ex2(s[2 * j] - m), p1 = ex2(s[2 * j + 1] - m);
                    sum += p0 + p1;
                    split_f16x2(p0, p1, ph[j], pl[j]);
                }
                sp_st_shared_f32(xsum_me + (G & 1) * 1024, sum);
                tmem_st_x16(tm + CF::tS + lane_addr + ch * 16, ph);
                tmem_st_x16(tm + CF::tS + lane_addr + 32 + ch * 16, pl);
                tmem_wait_st();
                tc_fence_before_sync();
                mbar_arrive(bars + CF::bPReady);
                tick(17);                                                        // 17: softmax
            }
        }
    } else {
        // =========================================================================================== QKV drain + normalisation
        // thread = token.  Iteration n: q, k, v of head n out of D_qkv (fp16 hi / lo: q -> TMEM, k and v -> shared memory),
        // O(n - 1) / rowsum -> fp16 hi / lo over O in TMEM (the projection's A operand).  Order inside an iteration, most
        // urgent first: q, k (S(n) is on the softmax chain) | v into registers (frees D_qkv) | normalisation of head n - 1
        // (the issuer's next projection) | v rows (P V(n) is a whole softmax away).
        sp_reg_inc<kSpRegsDr>();
        const int dw = warp - kSpDr0, r = dw * 32 + lane, wslot = r >> 6, tok = r & 63;
        const uint32_t lane_addr = static_cast<uint32_t>(dw * 32) << 16;
        const uint32_t rowoff = (tok >> 3) * 1024 + (tok & 7) * 128, sx = tok & 7;
        const uint32_t k_row = sb + CF::oK + wslot * 8192 + rowoff;
        const float* s_bq = reinterpret_cast<const float*>(smem + CF::oBq);
        const uint32_t xsum = sb + CF::oXch + 1024 + 4 * r;
        constexpr int NP = D / 2;                            // packed fp16 columns of a d-wide operand
        {                                                    // Q hi / lo columns incl. their pads start as zeros
            uint32_t z[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) z[j] = 0u;
            tmem_st_x32(tm + CF::tQ + lane_addr, z);
            tmem_wait_st();
        }
        auto st_operand = [&](uint32_t taddr, const uint32_t (&hi)[NP], const uint32_t (&lo)[NP]) {
            if constexpr (NP == 16) {
                tmem_st_x16(taddr, hi);
                tmem_st_x16(taddr + 16, lo);
            } else {
                static_assert(NP == 12 || NP == 16, "head dim 24 / 32");
                uint32_t a[8], b[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) { a[j] = hi[j]; b[j] = lo[j]; }
                tmem_st_x8(taddr, a);
                tmem_st_x4(taddr + 8, hi[8], hi[9], hi[10], hi[11]);
                tmem_st_x8(taddr + 16, b);
                tmem_st_x4(taddr + 24, lo[8], lo[9], lo[10], lo[11]);
            }
        };
        for (int n = 0; n <= total; ++n) {
            uint32_t raw[D];                                   // q, then k, then v columns of head n
            if (n < total) {
                const int h = n % H;
                mbar_wait(bars + CF::bDqFull, n & 1);
                tc_fence_after_sync();
                tick(24);                                                        // 24: wait D_qkv
#pragma unroll
                for (int c = 0; c < D / 8; ++c) {
                    uint32_t t8[8];
                    tmem_ld_x8(tm + CF::tDq + lane_addr + c * 8, t8);
#pragma unroll
                    for (int j = 0; j < 8; ++j) raw[c * 8 + j] = t8[j];
                }
                tmem_wait_ld();
                uint32_t qh[NP], ql[NP];
#pragma unroll
                for (int j = 0; j < NP; ++j)
                    split_f16x2(__uint_as_float(raw[2 * j]) + s_bq[h * D + 2 * j],
                                __uint_as_float(raw[2 * j + 1]) + s_bq[h * D + 2 * j + 1], qh[j], ql[j]);
#pragma unroll
                for (int c = 0; c < D / 8; ++c) {
                    uint32_t t8[8];
                    tmem_ld_x8(tm + CF::tDq + lane_addr + D + c * 8, t8);
#pragma unroll
                    for (int j = 0; j < 8; ++j) raw[c * 8 + j] = t8[j];
                }
                if (n > 0) mbar_wait(bars + CF::bQkFree, (n - 1) & 1);    // S(n - 1) has read Q and K
                tc_fence_after_sync();
                st_operand(tm + CF::tQ + lane_addr, qh, ql);
                tmem_wait_ld();
                tick(25);                                                        // 25: q -> TMEM (+ wait Q, K free)
#pragma unroll
                for (int ch = 0; ch < D / 8; ++ch) {           // k hi -> chunks 0.., k lo -> chunks 4..
                    uint32_t kh[4], kl[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        split_f16x2(__uint_as_float(raw[ch * 8 + 2 * j]), __uint_as_float(raw[ch * 8 + 2 * j + 1]), kh[j], kl[j]);
                    st_shared_v4(k_row + ((uint32_t(ch) ^ sx) << 4), kh[0], kh[1], kh[2], kh[3]);
                    st_shared_v4(k_row + ((uint32_t(4 + ch) ^ sx) << 4), kl[0], kl[1], kl[2], kl[3]);
                }
#pragma unroll
                for (int c = 0; c < D / 8; ++c) {
                    uint32_t t8[8];
                    tmem_ld_x8(tm + CF::tDq + lane_addr + 2 * D + c * 8, t8);
#pragma unroll
                    for (int j = 0; j < 8; ++j) raw[c * 8 + j] = t8[j];
                }
                tmem_wait_st();
                tc_fence_before_sync();
                fence_proxy_async_smem();
                mbar_arrive(bars + CF::bQkReady);
                tick(26);                                                        // 26: k -> shared memory
                tmem_wait_ld();
                tc_fence_before_sync();
                mbar_arrive(bars + CF::bDqEmpty);              // the accumulator may be overwritten by QKV(n + 1)
                tick(27);                                                        // 27: load v
            }
            if (n >= 1) {
                // O(n - 1) / rowsum first: the issuer needs it (projection) before it needs the v rows of head n
                const int G = n - 1;
                mbar_wait(bars + CF::bOFull, G & 1);
                tc_fence_after_sync();
                tick(29);                                                        // 29: wait O
                uint32_t oraw[D];
#pragma unroll
                for (int c = 0; c < D / 8; ++c) {
                    uint32_t t8[8];
                    tmem_ld_x8(tm + CF::tO + lane_addr + c * 8, t8);
#pragma unroll
                    for (int j = 0; j < 8; ++j) oraw[c * 8 + j] = t8[j];
                }
                const float inv = 1.0f / (sp_ld_shared_f32(xsum + (G & 1) * 1024) + sp_ld_shared_f32(xsum + (G & 1) * 1024 + 512));
                tmem_wait_ld();
                uint32_t oh[NP], ol[NP];
#pragma unroll
                for (int j = 0; j < NP; ++j)
                    split_f16x2(__uint_as_float(oraw[2 * j]) * inv, __uint_as_float(oraw[2 * j + 1]) * inv, oh[j], ol[j]);
                st_operand(tm + CF::tOA + lane_addr, oh, ol);
                if constexpr (NP == 12) {                        // k = 24 .. 31 of the projection operand: zeros
                    tmem_st_x4(tm + CF::tOA + lane_addr + 12, 0u, 0u, 0u, 0u);
                    tmem_st_x4(tm + CF::tOA + lane_addr + 28, 0u, 0u, 0u, 0u);
                }
                tmem_wait_st();
                tc_fence_before_sync();
                mbar_arrive(bars + CF::bOAReady);
                tick(30);                                                        // 30: normalisation
            }
            if (n < total) {
                // (O(n - 1) complete implies P V(n - 1) has read the V rows; the wait below then returns at once)
                if (n > 0) mbar_wait(bars + CF::bVFree, (n - 1) & 1);
#pragma unroll
                for (int ch = 0; ch < D / 8; ++ch) {           // v -> hi / lo rows [key][slot 0 d | slot 1 d]
                    uint32_t vh[4], vl[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        split_f16x2(__uint_as_float(raw[ch * 8 + 2 * j]), __uint_as_float(raw[ch * 8 + 2 * j + 1]), vh[j], vl[j]);
                    const uint32_t off = rowoff + ((uint32_t(wslot * (D / 8) + ch) ^ sx) << 4);
                    st_shared_v4(sb + CF::oVh + off, vh[0], vh[1], vh[2], vh[3]);
                    st_shared_v4(sb + CF::oVl + off, vl[0], vl[1], vl[2], vl[3]);
                }
                fence_proxy_async_smem();
                mbar_arrive(bars + CF::bVReady);
                tick(28);                                                        // 28: v -> shared memory
            }
        }
    }

    tc_fence_before_sync();
    __syncthreads();
    if (warp == kSpFeed) tmem_dealloc<512>(tm);
    if constexpr (kTiming) {      // per-CTA totals: [64 + cta] cycles, [64 + 256 + cta] tiles (buffer of 4096 u64)
        if (timing != nullptr && tid == 0) {
            timing[64 + blockIdx.x] = static_cast<unsigned long long>(clock64() - t_cta0);
            timing[64 + 256 + blockIdx.x] = my_tiles;
        }
    }
}

unsigned long long* g_sp_timing = nullptr;

typedef CUresult (*SpEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// 4-D tiled tensor map over the NCHW fp32 input, box = [16 ch][8][8]: one 16-channel slice of an 8 x 8 window
int sp_window_box_map(const float* x, int B, int C, int H, int W, CUtensorMap* map) {
    static SpEncodeTiledFn encode = nullptr;
    if (encode == nullptr) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        MWA_TRY_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres), "mwa_forward(tensor map)");
        if (fn == nullptr || qres != cudaDriverEntryPointSuccess) return MWA_ERR_UNSUPPORTED;
        encode = reinterpret_cast<SpEncodeTiledFn>(fn);
    }
    const cuuint64_t dims[4] = {cuuint64_t(W), cuuint64_t(H), cuuint64_t(C), cuuint64_t(B)};
    const cuuint64_t strides[3] = {cuuint64_t(W) * 4, cuuint64_t(H) * W * 4, cuuint64_t(C) * H * W * 4};
    const cuuint32_t box[4] = {8, 8, 16, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(x), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? MWA_OK : MWA_ERR_UNSUPPORTED;
}

template <class CF>
int launch_sp(const float* x, const float* alpha, float* out, const uint8_t* sp, int B, int H, int W, int shift,
              int32_t* kept_count, void* workspace, int64_t workspace_bytes, cudaStream_t st) {
    const Geom geo{B, H, W, shift, W / CF::WS, H / CF::WS, 0};
    return mwa_forward_lists<CF::WS>(x, alpha, out, geo, CF::C, kept_count, workspace, workspace_bytes, st,
                                     [&](int nwin, const int32_t* list, const int32_t* count) -> int {
        CUtensorMap x_map;
        memset(&x_map, 0, sizeof(x_map));
        const int rc = sp_window_box_map(x, B, CF::C, H, W, &x_map);
        if (rc != MWA_OK) return rc;
        const int smem = CF::oTotal;
        const int max_tiles = (nwin + 1) / 2;
        const int grid = max_tiles < kNumSMs ? max_tiles : kNumSMs;
        if (g_sp_timing != nullptr) {
            MWA_TRY_CUDA(cudaFuncSetAttribute(mwa_sp_kernel<CF, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem),
                         "mwa_forward(sp attr)");
            mwa_sp_kernel<CF, true><<<grid, kSpThreads, smem, st>>>(x, out, sp, list, count, geo, g_sp_timing, x_map);
        } else {
            MWA_TRY_CUDA(cudaFuncSetAttribute(mwa_sp_kernel<CF, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem),
                         "mwa_forward(sp attr)");
            mwa_sp_kernel<CF, false><<<grid, kSpThreads, smem, st>>>(x, out, sp, list, count, geo, nullptr, x_map);
        }
        return check_launch("mwa_forward(tcgen05 split precision)");
    });
}

}  // namespace

bool mwa_sp_supported(int C, int heads, int ws, int H, int W, int channels_last) {
    if (channels_last) return false;
    return C == 192 && ws == 8 && (heads == 8 || heads == 6) && H % 8 == 0 && W % 8 == 0 && W % 4 == 0;
}
int64_t mwa_sp_workspace_bytes(int64_t nwin) { return ListWs(nwin).total; }
void mwa_sp_set_timing_buffer(void* p) { g_sp_timing = static_cast<unsigned long long*>(p); }

void mwa_sp_prepare_images(const float* qkv_w, const float* qkv_b, const float* proj_w, const float* proj_b,
                           const float* table, int C, int heads, int ws, float scale, uint8_t* blk, cudaStream_t st) {
    const int64_t bytes = mwa_sp_section_bytes(C, heads, ws);
    if (bytes == 0) return;
    const MwaParamLayout L(C, heads, ws);
    uint8_t* dst = blk + L.img_sp;
    zero16_kernel<<<64, 256, 0, st>>>(reinterpret_cast<uint4*>(dst), bytes / 16);
    if (heads == 8) mwa_sp_prepare_kernel<SpCfg<8>><<<kNumSMs, 256, 0, st>>>(qkv_w, qkv_b, proj_w, proj_b, table, scale, dst);
    else mwa_sp_prepare_kernel<SpCfg<6>><<<kNumSMs, 256, 0, st>>>(qkv_w, qkv_b, proj_w, proj_b, table, scale, dst);
}

int mwa_forward_sp(const float* x, const float* alpha, float* out, const void* params, int B, int C, int H, int W,
                   int heads, int ws, int shift, int32_t* kept_count, void* workspace, int64_t workspace_bytes,
                   cudaStream_t st) {
    const MwaParamLayout L(C, heads, ws);
    const uint8_t* sp = static_cast<const uint8_t*>(params) + L.img_sp;
    if (heads == 8) return launch_sp<SpCfg<8>>(x, alpha, out, sp, B, H, W, shift, kept_count, workspace, workspace_bytes, st);
    if (heads == 6) return launch_sp<SpCfg<6>>(x, alpha, out, sp, B, H, W, shift, kept_count, workspace, workspace_bytes, st);
    return MWA_ERR_UNSUPPORTED;
}

}  // namespace b200
