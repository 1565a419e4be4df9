// Layout of the kernel-ready parameter blocks written by gdn_prepare / mwa_prepare.
// Host and device agree on the offsets through these structs (all offsets in bytes, 1024-byte aligned
// sections so that UMMA operand images can be bulk-copied straight into swizzled shared memory).
#pragma once
#include <stdint.h>

namespace b200 {

__host__ __device__ inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// ---------------------------------------------------------------- GDN
struct GdnParamLayout {
    int C, kblocks;
    int64_t beta;       // fp32 [C]            effective beta
    int64_t gamma;      // fp32 [C][C]         effective gamma, [out i][in j]
    int64_t gammaT;     // fp32 [C][C]         transposed, [in j][out i]
    int64_t mask_beta;  // uint8 [C]           1 where beta_p  >= beta_bound  (LowerBound pass-through, backward)
    int64_t mask_gamma; // uint8 [C][C]        1 where gamma_p >= gamma_bound
    int64_t img_hi;     // bf16 UMMA B-operand image of gamma (hi part): kblocks x [C rows x 64 k] K-major SW128
    int64_t img_lo;     // same for the lo part (gamma - hi)
    int64_t total;
    __host__ __device__ explicit GdnParamLayout(int C_) : C(C_), kblocks((C_ + 63) / 64) {
        int64_t o = 0;
        beta = o;       o = align_up(o + 4ll * C, 1024);
        gamma = o;      o = align_up(o + 4ll * C * C, 1024);
        gammaT = o;     o = align_up(o + 4ll * C * C, 1024);
        mask_beta = o;  o = align_up(o + C, 1024);
        mask_gamma = o; o = align_up(o + 1ll * C * C, 1024);
        const int64_t rows = align_up(C, 8);
        img_hi = o;     o = align_up(o + kblocks * rows * 128, 1024);
        img_lo = o;     o = align_up(o + kblocks * rows * 128, 1024);
        total = o;
    }
    __host__ __device__ int64_t img_bytes() const { return int64_t(kblocks) * align_up(C, 8) * 128; }
};

// ---------------------------------------------------------------- masked window attention
// size of the split-precision section (csrc/mwa_sp.cu, layout: SpParams<> there): per head the fp16 hi and lo
// K-major SW128 slabs of Wq|Wk|Wv per 64-channel K block as ring-slot sized elements, per head and output half the
// [hi | lo] slab of Wproj, the scaled q bias, the projection bias with the v bias folded in, the relative-position
// table times log2(e) and a 16 x 16 identity operand.  0 when the geometry is not covered.
__host__ __device__ inline int64_t mwa_sp_section_bytes(int C, int heads, int ws) {
    if (!(C == 192 && ws == 8 && (heads == 8 || heads == 6))) return 0;
    const int64_t tbl = (2 * ws - 1) * (2 * ws - 1);
    return int64_t(heads) * 3 * 2 * (3 * (C / heads) * 128) + int64_t(heads) * 2 * 12288 + 2 * int64_t(C) * 4 + align_up(heads * tbl * 4, 1024) + 2048;
}

struct MwaParamLayout {
    int C, heads, ws, N, d;
    int64_t header;     // float[4]: scale, -, -, -
    int64_t wqkvT;      // fp32 [C][3C]   qkv.weight transposed  ([in][out])
    int64_t bqkv;       // fp32 [3C]      (zeros when qkv_bias=False)
    int64_t wprojT;     // fp32 [C][C]    proj.weight transposed
    int64_t bproj;      // fp32 [C]
    int64_t bias;       // fp32 [heads][N][N]   expanded relative position bias
    int64_t img_sp;     // split-precision section (layout: SpParams<> in mwa_sp.cu)
    int64_t total;
    __host__ __device__ MwaParamLayout(int C_, int heads_, int ws_)
        : C(C_), heads(heads_), ws(ws_), N(ws_ * ws_), d(C_ / heads_) {
        int64_t o = 0;
        header = o;    o = align_up(o + 16, 1024);
        wqkvT = o;     o = align_up(o + 4ll * C * 3 * C, 1024);
        bqkv = o;      o = align_up(o + 4ll * 3 * C, 1024);
        wprojT = o;    o = align_up(o + 4ll * C * C, 1024);
        bproj = o;     o = align_up(o + 4ll * C, 1024);
        bias = o;      o = align_up(o + 4ll * heads * N * N, 1024);
        img_sp = o;    o = align_up(o + mwa_sp_section_bytes(C, heads, ws), 1024);
        total = o;
    }
};

}  // namespace b200
