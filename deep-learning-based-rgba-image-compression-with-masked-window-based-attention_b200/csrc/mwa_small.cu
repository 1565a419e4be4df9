// Masked window attention forward for SMALL windows (4 x 4 = 16 tokens) in plain fp32, sm_100a.
// Reference semantics: layers/masked_win_attention.py:169-251 (block), :96-131 (window attention) -- the reference's
// arithmetic is fp32 end to end, and so is this kernel: FFMA only, no tensor-core operand rounding anywhere, which is
// what the call sites need that feed the quantiser directly (enc.attention2 produces y, layers/TransformRGB.py:72-75).
// The model's configuration is C = 80, 8 heads of d = 10: too narrow for the tensor cores to pay (a 16 x 16 x 10 logit
// block per window and head), HBM-bound by its roofline (901 kFLOP and 10.3 kB per window), FFMA-bound in practice.
//
// Persistent CTAs of 256 threads; a group = 4 kept windows = 64 tokens:
//   gather   x of the group -> Xt[c][token] in shared memory (also the residual, exact)
//   QKV      [64 x C] x [C x 3C] register-tiled: thread = 4 tokens (one window row) x 3C/16 outputs, weights resident in
//            shared memory (padded to 16-float groups so that every operand read is one LDS.128)
//   core     thread = (window, head, 2 query rows): 16 logits per row in registers, + relative-position bias
//            (+ SW-MSA region mask), softmax, P V -- no shuffles, no barriers inside
//   proj     [64 x C] x [C x C]: thread = 4 tokens x C/16 outputs, + bias + residual, float2 stores (a window row)
// Dropped windows are copied through by mwa_copy_dropped_kernel (only the dropped ones).
#include "mwa_lists.cuh"

namespace b200 {
namespace {

template <int C_, int HEADS_>
struct SmallCfg {
    static constexpr int C = C_, HEADS = HEADS_, D = C / HEADS, WS = 4, N = 16, GW = 4, T = GW * N;   // 64 tokens per group
    static_assert(C % 16 == 0 && C % HEADS == 0, "C must be a multiple of 16 and of the head count");
    static constexpr int QO = 3 * C / 16, PO = C / 16;       // outputs per thread: QKV, projection
    static_assert(QO <= 16 && PO <= 8, "per-thread tile too large");
    static constexpr int LDQ = 3 * C + 1;                    // row stride of the q | k | v tile (odd: conflict-free columns)
    // shared memory (floats)
    static constexpr int oXt = 0;                            // [C][T]      x, transposed (token fastest)
    static constexpr int oOt = oXt + C * T;                  // [C][T]      attention output, transposed
    static constexpr int oQkv = oOt + C * T;                 // [T][LDQ]
    static constexpr int oWq = (oQkv + T * LDQ + 3) / 4 * 4; // [C][16][16] Wqkv^T, output group og at [..][og][0 .. QO)
    static constexpr int oWp = oWq + C * 256;                // [C][C]      Wproj^T
    static constexpr int oBq = oWp + C * C;                // [3C] qkv bias (q part pre-scaled)
    static constexpr int oBp = oBq + 3 * C;                  // [C]
    static constexpr int oBias = oBp + C;                    // [HEADS][N][N]
    static constexpr int oReg = oBias + HEADS * N * N;       // [T] region id of each token (int)
    static constexpr int total = oReg + T;
    static_assert(total * 4 <= 227 * 1024, "shared memory budget");
};

template <class CF>
__global__ void __launch_bounds__(256, 1)
mwa_small_kernel(const float* __restrict__ x, float* __restrict__ out, const uint8_t* __restrict__ blk,
                 const int32_t* __restrict__ list, const int32_t* __restrict__ count_p, Geom geo) {
    constexpr int C = CF::C, H = CF::HEADS, D = CF::D, WS = CF::WS, N = CF::N, T = CF::T, QO = CF::QO, PO = CF::PO,
                  LDQ = CF::LDQ;
    extern __shared__ __align__(16) float sm[];
    float* Xt = sm + CF::oXt;
    float* Ot = sm + CF::oOt;
    float* Qkv = sm + CF::oQkv;
    float* Wq = sm + CF::oWq;
    float* Wp = sm + CF::oWp;
    float* Bq = sm + CF::oBq;
    float* Bp = sm + CF::oBp;
    float* Bias = sm + CF::oBias;
    int* Reg = reinterpret_cast<int*>(sm + CF::oReg);
    const int tid = threadIdx.x;
    const MwaParamLayout L(C, H, WS);
    const float scale = reinterpret_cast<const float*>(blk + L.header)[0];

    // ---- parameters -> shared memory, once per CTA
    {
        const float* wqkvT = reinterpret_cast<const float*>(blk + L.wqkvT);       // [C][3C]
        for (int e = tid; e < C * 256; e += 256) {
            const int k = e >> 8, og = (e >> 4) & 15, j = e & 15;
            const int o = og * QO + j;
            Wq[e] = (j < QO) ? wqkvT[k * 3 * C + o] * (o < C ? scale : 1.0f) : 0.f;
        }
        const float* wprojT = reinterpret_cast<const float*>(blk + L.wprojT);     // [C][C]
        for (int e = tid; e < C * C; e += 256) Wp[e] = wprojT[e];
        const float* bqkv = reinterpret_cast<const float*>(blk + L.bqkv);
        for (int e = tid; e < 3 * C; e += 256) Bq[e] = bqkv[e] * (e < C ? scale : 1.0f);
        const float* bproj = reinterpret_cast<const float*>(blk + L.bproj);
        for (int e = tid; e < C; e += 256) Bp[e] = bproj[e];
        const float* bias = reinterpret_cast<const float*>(blk + L.bias);
        for (int e = tid; e < H * N * N; e += 256) Bias[e] = bias[e];
    }
    __syncthreads();

    const int count = *count_p;
    const int ngroups = (count + CF::GW - 1) / CF::GW;
    const int64_t hw = int64_t(geo.H) * geo.W;
    const int tg = tid & 15, og = tid >> 4;                 // GEMM roles: token group (one window row) x output group
    const bool vec2 = (geo.shift % 2 == 0) && (geo.W % 2 == 0);

    for (int grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
        // ---- gather: Xt[c][w * 16 + r * 4 + px]; thread = (window slot, row, channel stripe)
        {
            const int w = tid & 3, r = (tid >> 2) & 3, cs = tid >> 4;           // 16 channel stripes
            const int lidx = grp * CF::GW + w;
            const bool valid = lidx < count;
            int b = 0, wy = 0, wx = 0;
            if (valid) window_coords(geo, list[lidx], b, wy, wx);
            int py = wy * WS + r + geo.shift, px0 = wx * WS + geo.shift;
            if (py >= geo.H) py -= geo.H;
            if (px0 >= geo.W) px0 -= geo.W;
            const bool wrap = px0 + WS > geo.W;                                  // the row wraps round the right border
            const float* src = x + int64_t(b) * C * hw + int64_t(py) * geo.W;
            float* dst = Xt + w * 16 + r * 4;
            for (int c = cs; c < C; c += 16) {
                float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
                if (valid) {
                    const float* p = src + int64_t(c) * hw;
                    if (vec2 && !wrap) {
                        const float2 a = __ldg(reinterpret_cast<const float2*>(p + px0));
                        const float2 bb = __ldg(reinterpret_cast<const float2*>(p + px0 + 2));
                        v0 = a.x; v1 = a.y; v2 = bb.x; v3 = bb.y;
                    } else {
                        int q0 = px0, q1 = px0 + 1, q2 = px0 + 2, q3 = px0 + 3;
                        if (q1 >= geo.W) q1 -= geo.W;
                        if (q2 >= geo.W) q2 -= geo.W;
                        if (q3 >= geo.W) q3 -= geo.W;
                        v0 = __ldg(p + q0); v1 = __ldg(p + q1); v2 = __ldg(p + q2); v3 = __ldg(p + q3);
                    }
                }
                *reinterpret_cast<float4*>(dst + c * T) = make_float4(v0, v1, v2, v3);
            }
            if (cs == 0) {
                // SW-MSA region id of this row's four tokens in the shifted frame (layers/masked_win_attention.py:194-216)
                const int ys = wy * WS + r;
                const int by = (ys >= geo.H - WS) + (ys >= geo.H - geo.shift);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int xs = wx * WS + i;
                    const int bx = (xs >= geo.W - WS) + (xs >= geo.W - geo.shift);
                    Reg[w * 16 + r * 4 + i] = (geo.shift > 0) ? 3 * by + bx : 0;
                }
            }
        }
        __syncthreads();

        // ---- QKV: Qkv[t][o] = sum_k Xt[k][t] Wq[k][o] + b   (q columns and bias pre-scaled, :103-106)
        {
            float acc[4][QO];
#pragma unroll
            for (int j = 0; j < QO; ++j) {
                const float bv = Bq[og * QO + j];
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[i][j] = bv;
            }
            const float* xp = Xt + tg * 4;
            const float* wp = Wq + og * 16;
#pragma unroll 4
            for (int k = 0; k < C; ++k) {
                const float4 xv = *reinterpret_cast<const float4*>(xp + k * T);
                float wv[16];
#pragma unroll
                for (int j4 = 0; j4 < (QO + 3) / 4; ++j4)
                    *reinterpret_cast<float4*>(wv + 4 * j4) = *reinterpret_cast<const float4*>(wp + k * 256 + 4 * j4);
#pragma unroll
                for (int j = 0; j < QO; ++j) {
                    acc[0][j] = fmaf(xv.x, wv[j], acc[0][j]);
                    acc[1][j] = fmaf(xv.y, wv[j], acc[1][j]);
                    acc[2][j] = fmaf(xv.z, wv[j], acc[2][j]);
                    acc[3][j] = fmaf(xv.w, wv[j], acc[3][j]);
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < QO; ++j) Qkv[(tg * 4 + i) * LDQ + og * QO + j] = acc[i][j];
        }
        __syncthreads();

        // ---- attention core: work item = (window slot w, head h, row pair): GW * H * 8 items
        for (int item = tid; item < CF::GW * H * 8; item += 256) {
            const int rp = item & 7, h = (item >> 3) % H, w = item / (8 * H);
            const int t0 = w * 16;
            float s[2][16];
#pragma unroll
            for (int a = 0; a < 2; ++a) {
                const int i = rp * 2 + a;
                float q[D];
#pragma unroll
                for (int c = 0; c < D; ++c) q[c] = Qkv[(t0 + i) * LDQ + h * D + c];
                const float* bh = Bias + (h * N + i) * N;
                const int ri = Reg[t0 + i];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float* kp = Qkv + (t0 + j) * LDQ + C + h * D;
                    float d = 0.f;
#pragma unroll
                    for (int c = 0; c < D; ++c) d = fmaf(q[c], kp[c], d);
                    d += bh[j];
                    if (Reg[t0 + j] != ri) d += kNegMask;
                    s[a][j] = d;
                }
            }
#pragma unroll
            for (int a = 0; a < 2; ++a) {
                float m = s[a][0];
#pragma unroll
                for (int j = 1; j < 16; ++j) m = fmaxf(m, s[a][j]);
                float sum = 0.f;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    s[a][j] = __expf(s[a][j] - m);
                    sum += s[a][j];
                }
                const float inv = 1.0f / sum;
                float o[D];
#pragma unroll
                for (int c = 0; c < D; ++c) o[c] = 0.f;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float* vp = Qkv + (t0 + j) * LDQ + 2 * C + h * D;
#pragma unroll
                    for (int c = 0; c < D; ++c) o[c] = fmaf(s[a][j], vp[c], o[c]);
                }
#pragma unroll
                for (int c = 0; c < D; ++c) Ot[(h * D + c) * T + t0 + rp * 2 + a] = o[c] * inv;
            }
        }
        __syncthreads();

        // ---- projection + bias + residual, stored to the un-shifted position   (:129, :237-249)
        {
            float acc[4][PO];
#pragma unroll
            for (int j = 0; j < PO; ++j) {
                const float bv = Bp[og * PO + j];
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[i][j] = bv;
            }
            const float* op = Ot + tg * 4;
            const float* wp = Wp + og * PO;
#pragma unroll 4
            for (int k = 0; k < C; ++k) {
                const float4 ov = *reinterpret_cast<const float4*>(op + k * T);
                float wv[PO];
#pragma unroll
                for (int j = 0; j < PO; ++j) wv[j] = wp[k * C + j];
#pragma unroll
                for (int j = 0; j < PO; ++j) {
                    acc[0][j] = fmaf(ov.x, wv[j], acc[0][j]);
                    acc[1][j] = fmaf(ov.y, wv[j], acc[1][j]);
                    acc[2][j] = fmaf(ov.z, wv[j], acc[2][j]);
                    acc[3][j] = fmaf(ov.w, wv[j], acc[3][j]);
                }
            }
            const int w = tg >> 2, r = tg & 3;
            const int lidx = grp * CF::GW + w;
            if (lidx < count) {
                int b, wy, wx;
                window_coords(geo, list[lidx], b, wy, wx);
                int py = wy * WS + r + geo.shift, px0 = wx * WS + geo.shift;
                if (py >= geo.H) py -= geo.H;
                if (px0 >= geo.W) px0 -= geo.W;
                const bool wrap = px0 + WS > geo.W;
                float* dst = out + int64_t(b) * C * hw + int64_t(py) * geo.W;
#pragma unroll
                for (int j = 0; j < PO; ++j) {
                    const int c = og * PO + j;
                    const float4 xv = *reinterpret_cast<const float4*>(Xt + c * T + tg * 4);
                    const float y0 = xv.x + acc[0][j], y1 = xv.y + acc[1][j], y2 = xv.z + acc[2][j], y3 = xv.w + acc[3][j];
                    float* p = dst + int64_t(c) * hw;
                    if (vec2 && !wrap) {
                        *reinterpret_cast<float2*>(p + px0) = make_float2(y0, y1);
                        *reinterpret_cast<float2*>(p + px0 + 2) = make_float2(y2, y3);
                    } else {
                        int q1 = px0 + 1, q2 = px0 + 2, q3 = px0 + 3;
                        if (q1 >= geo.W) q1 -= geo.W;
                        if (q2 >= geo.W) q2 -= geo.W;
                        if (q3 >= geo.W) q3 -= geo.W;
                        p[px0] = y0; p[q1] = y1; p[q2] = y2; p[q3] = y3;
                    }
                }
            }
        }
        __syncthreads();
    }
}

template <class CF>
int launch_small(const float* x, const float* alpha, float* out, const uint8_t* params, int B, int H, int W, int shift,
                 int32_t* kept_count, void* workspace, int64_t workspace_bytes, cudaStream_t st) {
    const Geom geo{B, H, W, shift, W / CF::WS, H / CF::WS, 0};
    return mwa_forward_lists<CF::WS>(x, alpha, out, geo, CF::C, kept_count, workspace, workspace_bytes, st,
                                     [&](int nwin, const int32_t* list, const int32_t* count) -> int {
        const int smem = CF::total * 4;
        MWA_TRY_CUDA(cudaFuncSetAttribute(mwa_small_kernel<CF>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem),
                     "mwa_forward(small attr)");
        const int max_groups = (nwin + CF::GW - 1) / CF::GW;
        const int grid = max_groups < kNumSMs ? max_groups : kNumSMs;
        mwa_small_kernel<CF><<<grid, 256, smem, st>>>(x, out, params, list, count, geo);
        return check_launch("mwa_forward(fp32 small windows)");
    });
}

}  // namespace

bool mwa_small_supported(int C, int heads, int ws, int channels_last) {
    return !channels_last && ws == 4 && C == 80 && heads == 8;
}
int64_t mwa_small_workspace_bytes(int64_t nwin) { return ListWs(nwin).total; }

int mwa_forward_small(const float* x, const float* alpha, float* out, const void* params, int B, int C, int H, int W,
                      int heads, int ws, int shift, int32_t* kept_count, void* workspace, int64_t workspace_bytes,
                      cudaStream_t st) {
    if (!mwa_small_supported(C, heads, ws, 0)) return MWA_ERR_UNSUPPORTED;
    return launch_small<SmallCfg<80, 8>>(x, alpha, out, static_cast<const uint8_t*>(params), B, H, W, shift, kept_count,
                                         workspace, workspace_bytes, st);
}

}  // namespace b200
