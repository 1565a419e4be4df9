// Masked window attention: parameter preparation and the general-shape SIMT forward kernel.
// Reference semantics: layers/masked_win_attention.py:169-251 (block), :96-131 (window attention),
// :35-47 (keep predicate), :194-216 (SW-MSA region mask); layers/win_attention.py:153-207 (alpha == NULL).
// The forwards for the model's configurations live in mwa_sp.cu (8x8 windows, C = 192) and mwa_small.cu (4x4, C = 80).
#include "common.cuh"
#include "params.cuh"
#include "status.cuh"

namespace b200 {

int mwa_forward_sp(const float* x, const float* alpha, float* out, const void* params, int B, int C, int H, int W,
                   int heads, int ws, int shift, int32_t* kept_count, void* workspace, int64_t workspace_bytes,
                   cudaStream_t st);                                                                          // mwa_sp.cu
bool mwa_sp_supported(int C, int heads, int ws, int H, int W, int channels_last);
int64_t mwa_sp_workspace_bytes(int64_t nwin);
void mwa_sp_set_timing_buffer(void* p);
void mwa_sp_prepare_images(const float* qkv_w, const float* qkv_b, const float* proj_w, const float* proj_b,
                           const float* table, int C, int heads, int ws, float scale, uint8_t* blk, cudaStream_t st);

int mwa_forward_small(const float* x, const float* alpha, float* out, const void* params, int B, int C, int H, int W,
                      int heads, int ws, int shift, int32_t* kept_count, void* workspace, int64_t workspace_bytes,
                      cudaStream_t st);                                                                       // mwa_small.cu
bool mwa_small_supported(int C, int heads, int ws, int channels_last);
int64_t mwa_small_workspace_bytes(int64_t nwin);

namespace {

constexpr int kThreads = 256;
constexpr float kNegMask = -100.0f;                 // layers/masked_win_attention.py:214

// ------------------------------------------------------------------ prepare
__global__ void mwa_prepare_kernel(const float* __restrict__ qkv_w, const float* __restrict__ qkv_b,
                                   const float* __restrict__ proj_w, const float* __restrict__ proj_b,
                                   const float* __restrict__ table, int C, int heads, int ws, float scale,
                                   uint8_t* __restrict__ blk) {
    const MwaParamLayout L(C, heads, ws);
    float* hdr = reinterpret_cast<float*>(blk + L.header);
    float* wqkvT = reinterpret_cast<float*>(blk + L.wqkvT);
    float* bqkv = reinterpret_cast<float*>(blk + L.bqkv);
    float* wprojT = reinterpret_cast<float*>(blk + L.wprojT);
    float* bproj = reinterpret_cast<float*>(blk + L.bproj);
    float* bias = reinterpret_cast<float*>(blk + L.bias);
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int nth = gridDim.x * blockDim.x;
    if (tid == 0) {
        hdr[0] = scale;
        hdr[1] = hdr[2] = hdr[3] = 0.f;
    }
    for (int e = tid; e < 3 * C * C; e += nth) {           // qkv.weight (3C, C) -> [C][3C]
        const int o = e / C, c = e % C;
        wqkvT[int64_t(c) * 3 * C + o] = qkv_w[e];
    }
    for (int e = tid; e < 3 * C; e += nth) bqkv[e] = qkv_b ? qkv_b[e] : 0.f;
    for (int e = tid; e < C * C; e += nth) {
        const int o = e / C, c = e % C;
        wprojT[int64_t(c) * C + o] = proj_w[e];
    }
    for (int e = tid; e < C; e += nth) bproj[e] = proj_b[e];
    const int N = ws * ws;
    for (int e = tid; e < heads * N * N; e += nth) {       // expanded relative position bias [h][i][j]
        const int h = e / (N * N), i = (e / N) % N, j = e % N;
        const int dy = i / ws - j / ws + ws - 1, dx = i % ws - j % ws + ws - 1;
        bias[e] = table[(dy * (2 * ws - 1) + dx) * heads + h];
    }
}

// ------------------------------------------------------------------ geometry helpers
struct Geo {
    int B, C, H, W, ws, shift, nwx, nwy, N;
    int channels_last;
    int tokens;          // 1: x/out are (K, N, C) window tokens (WindowAttention.forward), no geometry, no residual
    int mask_nw;         // tokens mode: number of windows in the external additive mask (0 = none)
    // token t of window (wy, wx): shifted-frame coords and original pixel
    __device__ __forceinline__ void token_pixel(int wy, int wx, int t, int& y, int& x) const {
        int ys = wy * ws + t / ws, xs = wx * ws + t % ws;
        y = ys + shift; if (y >= H) y -= H;
        x = xs + shift; if (x >= W) x -= W;
    }
    __device__ __forceinline__ int region(int wy, int wx, int t) const {   // SW-MSA region id in the shifted frame
        const int ys = wy * ws + t / ws, xs = wx * ws + t % ws;
        const int by = (ys >= H - ws) + (ys >= H - shift), bx = (xs >= W - ws) + (xs >= W - shift);
        return 3 * by + bx;
    }
    __device__ __forceinline__ int64_t offset(int b, int c, int y, int x) const {
        return channels_last ? ((int64_t(b) * H + y) * W + x) * C + c : ((int64_t(b) * C + c) * H + y) * W + x;
    }
    // element (token t, channel c) of window `win` = (b, wy, wx)
    __device__ __forceinline__ int64_t elem(int win, int b, int wy, int wx, int t, int c) const {
        if (tokens) return (int64_t(win) * N + t) * C + c;
        int y, xx;
        token_pixel(wy, wx, t, y, xx);
        return offset(b, c, y, xx);
    }
};

// out[n][o] = sum_k A[n][k] * WT[k][o] + bias[o]   for n < N, o < O;  A in smem (row stride lda), WT global [K][O].
// work item = (output column o, chunk of TN tokens); lanes run over o -> coalesced weight reads, broadcast A reads.
template <int TN, class Epilogue>
__device__ __forceinline__ void gemm_tokens(const float* __restrict__ A, int lda, const float* __restrict__ WT,
                                            const float* __restrict__ bias, int N, int O, int K, Epilogue epi) {
    const int nchunks = (N + TN - 1) / TN;
    for (int item = threadIdx.x; item < O * nchunks; item += kThreads) {
        const int o = item % O, n0 = (item / O) * TN;
        float acc[TN];
        const float b = bias[o];
#pragma unroll
        for (int i = 0; i < TN; ++i) acc[i] = b;
        for (int k = 0; k < K; k += 4) {
            float w[4];
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) w[kk] = (k + kk < K) ? __ldg(WT + int64_t(k + kk) * O + o) : 0.f;
#pragma unroll
            for (int i = 0; i < TN; ++i) {
                if (n0 + i < N) {
                    const float* a = A + (n0 + i) * lda + k;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        if (k + kk < K) acc[i] = fmaf(a[kk], w[kk], acc[i]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < TN; ++i)
            if (n0 + i < N) epi(n0 + i, o, acc[i]);
    }
}

// ------------------------------------------------------------------ SIMT forward: one CTA per window
// smem: xw[N][C] (later reused for the head-concatenated attention output), qkv[N][3C+1], S[N][N+1], flag
__global__ void __launch_bounds__(kThreads)
mwa_simt_kernel(const float* __restrict__ x, const float* __restrict__ alpha, float* __restrict__ out,
                const uint8_t* __restrict__ blk, Geo g, int heads, int32_t* __restrict__ kept_count,
                const float* __restrict__ ext_mask) {
    extern __shared__ float smem[];
    const int C = g.C, N = g.N, ws = g.ws;
    const int d = C / heads;
    const int ldq = 3 * C + 1, lds = N + 1;
    float* xw = smem;                       // N * C
    float* qkv = xw + N * C;                // N * ldq
    float* S = qkv + N * ldq;               // N * lds
    __shared__ float red[kThreads / 32];
    __shared__ int keep_s;

    const MwaParamLayout L(C, heads, ws);
    const float scale = reinterpret_cast<const float*>(blk + L.header)[0];
    const float* wqkvT = reinterpret_cast<const float*>(blk + L.wqkvT);
    const float* bqkv = reinterpret_cast<const float*>(blk + L.bqkv);
    const float* wprojT = reinterpret_cast<const float*>(blk + L.wprojT);
    const float* bproj = reinterpret_cast<const float*>(blk + L.bproj);
    const float* bias = reinterpret_cast<const float*>(blk + L.bias);

    const int tid = threadIdx.x;
    const int win = blockIdx.x;
    const int b = win / (g.nwy * g.nwx), wy = (win / g.nwx) % g.nwy, wx = win % g.nwx;
    const bool c_fast = g.channels_last || g.tokens;          // iteration order that coalesces global accesses

    // ---- keep predicate: sum of the window's alpha != 0   (fp32 sum; order-free for alpha >= 0)
    bool keep = true;
    if (alpha != nullptr) {
        float a = 0.f;
        for (int t = tid; t < N; t += kThreads) {
            int y, xx;
            g.token_pixel(wy, wx, t, y, xx);
            a += __ldg(alpha + (int64_t(b) * g.H + y) * g.W + xx);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
        if ((tid & 31) == 0) red[tid >> 5] = a;
        __syncthreads();
        if (tid == 0) {
            float tot = 0.f;
            for (int i = 0; i < kThreads / 32; ++i) tot += red[i];
            keep_s = (tot != 0.f);
        }
        __syncthreads();
        keep = keep_s != 0;
    }
    if (kept_count != nullptr && tid == 0 && keep) atomicAdd(kept_count, 1);

    if (!keep) {                            // dropped window: the block is the identity there
        for (int e = tid; e < N * C; e += kThreads) {
            const int c = c_fast ? e % C : e / N, t = c_fast ? e / C : e % N;
            const int64_t off = g.elem(win, b, wy, wx, t, c);
            out[off] = __ldg(x + off);
        }
        return;
    }

    // ---- gather the window: xw[t][c]
    for (int e = tid; e < N * C; e += kThreads) {
        const int c = c_fast ? e % C : e / N, t = c_fast ? e / C : e % N;
        xw[t * C + c] = __ldg(x + g.elem(win, b, wy, wx, t, c));
    }
    __syncthreads();

    // ---- qkv = xw * Wqkv^T + b ; q pre-scaled   (layers/masked_win_attention.py:103-106)
    gemm_tokens<16>(xw, C, wqkvT, bqkv, N, 3 * C, C, [&](int n, int o, float v) {
        qkv[n * ldq + o] = (o < C) ? v * scale : v;
    });
    __syncthreads();

    // ---- per head: S = q k^T + bias (+ region mask) ; softmax ; O_h = P v_h  -> xw[:, h*d : (h+1)*d]
    for (int h = 0; h < heads; ++h) {
        const float* bh = bias + int64_t(h) * N * N;
        for (int e = tid; e < N * N; e += kThreads) {
            const int i = e / N, j = e % N;
            const float* q = qkv + i * ldq + h * d;
            const float* k = qkv + j * ldq + C + h * d;
            float acc = 0.f;
            for (int c = 0; c < d; ++c) acc = fmaf(q[c], k[c], acc);
            acc += __ldg(bh + e);
            if (g.tokens) {
                if (g.mask_nw > 0) acc += __ldg(ext_mask + (int64_t(win % g.mask_nw) * N + i) * N + j);
            } else if (g.shift > 0 && g.region(wy, wx, i) != g.region(wy, wx, j)) {
                acc += kNegMask;
            }
            S[i * lds + j] = acc;
        }
        __syncthreads();
        for (int i = tid >> 5; i < N; i += kThreads / 32) {          // warp per row
            float* row = S + i * lds;
            float m = -INFINITY;
            for (int j = tid & 31; j < N; j += 32) m = fmaxf(m, row[j]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            float sum = 0.f;
            for (int j = tid & 31; j < N; j += 32) {
                const float e = expf(row[j] - m);
                row[j] = e;
                sum += e;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            const float inv = 1.f / sum;
            for (int j = tid & 31; j < N; j += 32) row[j] *= inv;
        }
        __syncthreads();
        for (int e = tid; e < N * d; e += kThreads) {
            const int i = e / d, c = e % d;
            const float* p = S + i * lds;
            const float* v = qkv + 2 * C + h * d + c;
            float acc = 0.f;
            for (int j = 0; j < N; ++j) acc = fmaf(p[j], v[j * ldq], acc);
            xw[i * C + h * d + c] = acc;
        }
        __syncthreads();
    }

    // ---- proj + residual, scattered back to the un-shifted position   (:129, :237-249)
    gemm_tokens<16>(xw, C, wprojT, bproj, N, C, C, [&](int n, int o, float v) {
        qkv[n * ldq + o] = v;               // stage: qkv buffer is free now
    });
    __syncthreads();
    for (int e = tid; e < N * C; e += kThreads) {
        const int c = c_fast ? e % C : e / N, t = c_fast ? e / C : e % N;
        const int64_t off = g.elem(win, b, wy, wx, t, c);
        out[off] = g.tokens ? qkv[t * ldq + c] : __ldg(x + off) + qkv[t * ldq + c];
    }
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" {

int64_t mwa_param_bytes(int C, int heads, int ws) {
    if (C <= 0 || heads <= 0 || ws <= 0 || C % heads != 0) return MWA_ERR_INVALID;
    return MwaParamLayout(C, heads, ws).total;
}

int mwa_prepare(const float* qkv_w, const float* qkv_b, const float* proj_w, const float* proj_b,
                const float* bias_table, int C, int heads, int ws, float scale, void* params, int64_t params_bytes,
                void* stream) {
    if (!qkv_w || !proj_w || !proj_b || !bias_table || !params) return MWA_ERR_INVALID;
    if (C <= 0 || heads <= 0 || ws <= 0 || C % heads != 0) return MWA_ERR_INVALID;
    if (!aligned16(params)) return MWA_ERR_ALIGNMENT;
    const MwaParamLayout L(C, heads, ws);
    if (params_bytes < L.total) return MWA_ERR_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint8_t* blk = static_cast<uint8_t*>(params);
    mwa_prepare_kernel<<<148, 256, 0, st>>>(qkv_w, qkv_b, proj_w, proj_b, bias_table, C, heads, ws, scale, blk);
    const int rc = check_launch("mwa_prepare");
    if (rc != MWA_OK) return rc;
    mwa_sp_prepare_images(qkv_w, qkv_b, proj_w, proj_b, bias_table, C, heads, ws, scale, blk, st);
    return check_launch("mwa_prepare(split-precision images)");
}

void mwa_debug_set_timing_buffer(void* device_u64x8192) { mwa_sp_set_timing_buffer(device_u64x8192); }

int64_t mwa_workspace_bytes(int B, int H, int W, int ws) {
    if (B < 0 || H <= 0 || W <= 0 || ws <= 0) return MWA_ERR_INVALID;
    const int64_t nwin = int64_t(B) * (H / ws) * (W / ws);
    const int64_t a = mwa_sp_workspace_bytes(nwin), b = mwa_small_workspace_bytes(nwin);
    return a > b ? a : b;
}

int mwa_fast_path_needs_nchw(int C, int heads, int ws) {
    return (mwa_sp_supported(C, heads, ws, 8, 8, 0) || mwa_small_supported(C, heads, ws, 0)) ? 1 : 0;
}

int mwa_forward(const float* x, const float* alpha, float* out, const void* params, int B, int C, int H, int W,
                int heads, int ws, int shift, int channels_last, int algo, int32_t* kept_count, void* workspace,
                int64_t workspace_bytes, void* stream) {
    if (B < 0 || C <= 0 || H <= 0 || W <= 0 || heads <= 0 || ws <= 0 || C % heads != 0) return MWA_ERR_INVALID;
    if (shift < 0 || shift >= ws) return MWA_ERR_INVALID;
    if (H % ws != 0 || W % ws != 0) return MWA_ERR_INVALID;
    if (algo != MWA_ALGO_AUTO && algo != MWA_ALGO_SIMT && algo != MWA_ALGO_TCGEN05) return MWA_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (kept_count) MWA_TRY_CUDA(cudaMemsetAsync(kept_count, 0, sizeof(int32_t), st), "mwa_forward(memset)");
    if (B == 0) return MWA_OK;                              // empty batch: x / out may be null
    if (!x || !out || !params) return MWA_ERR_INVALID;
    // MWA_ALGO_AUTO is fp32-faithful on every shape (the reference's arithmetic is fp32 end to end):
    //   8x8 windows, C = 192: split-precision tcgen05 kernel (every operand fp16 hi + lo, three passes);
    //   4x4 windows, C = 80:  plain fp32 kernel for small windows;
    //   anything else:        the general fp32 SIMT kernel.
    // MWA_ALGO_TCGEN05 asks for the split-precision kernel and fails where it does not cover the shape.
    if ((algo == MWA_ALGO_AUTO || algo == MWA_ALGO_TCGEN05) && mwa_sp_supported(C, heads, ws, H, W, channels_last)) {
        if (!aligned16(x) || !aligned16(out)) return MWA_ERR_ALIGNMENT;
        return mwa_forward_sp(x, alpha, out, params, B, C, H, W, heads, ws, shift, kept_count, workspace, workspace_bytes, st);
    }
    if (algo == MWA_ALGO_AUTO && mwa_small_supported(C, heads, ws, channels_last)) {
        if (!aligned16(x) || !aligned16(out)) return MWA_ERR_ALIGNMENT;
        return mwa_forward_small(x, alpha, out, params, B, C, H, W, heads, ws, shift, kept_count, workspace, workspace_bytes,
                                 st);
    }
    if (algo == MWA_ALGO_TCGEN05) return MWA_ERR_UNSUPPORTED;
    const int N = ws * ws;
    if (N > 64) return MWA_ERR_UNSUPPORTED;
    const int64_t smem = 4ll * (int64_t(N) * C + int64_t(N) * (3 * C + 1) + int64_t(N) * (N + 1));
    if (smem > 227 * 1024 - 64) return MWA_ERR_UNSUPPORTED;
    const int64_t nwin = int64_t(B) * (H / ws) * (W / ws);
    if (nwin > 0x7fffffffll) return MWA_ERR_UNSUPPORTED;
    Geo g{B, C, H, W, ws, shift, W / ws, H / ws, N, channels_last, 0, 0};
    MWA_TRY_CUDA(cudaFuncSetAttribute(mwa_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)),
                 "mwa_forward(simt attr)");
    mwa_simt_kernel<<<static_cast<unsigned>(nwin), kThreads, smem, st>>>(x, alpha, out,
                                                                         static_cast<const uint8_t*>(params), g, heads,
                                                                         kept_count, nullptr);
    return check_launch("mwa_forward(simt)");
}

int window_attention_forward(const float* xw, const float* mask, float* out, const void* params, int64_t K, int C,
                             int heads, int ws, int mask_windows, void* stream) {
    if (!xw || !out || !params) return MWA_ERR_INVALID;
    if (K < 0 || C <= 0 || heads <= 0 || ws <= 0 || C % heads != 0 || mask_windows < 0) return MWA_ERR_INVALID;
    if (mask_windows > 0 && (!mask || K % mask_windows != 0)) return MWA_ERR_INVALID;
    if (K == 0) return MWA_OK;
    const int N = ws * ws;
    if (N > 64 || K > 0x7fffffffll) return MWA_ERR_UNSUPPORTED;
    const int64_t smem = 4ll * (int64_t(N) * C + int64_t(N) * (3 * C + 1) + int64_t(N) * (N + 1));
    if (smem > 227 * 1024 - 64) return MWA_ERR_UNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Geo g{static_cast<int>(K), C, ws, ws, ws, 0, 1, 1, N, 1, 1, mask_windows};
    MWA_TRY_CUDA(cudaFuncSetAttribute(mwa_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)),
                 "window_attention_forward(attr)");
    mwa_simt_kernel<<<static_cast<unsigned>(K), kThreads, smem, st>>>(xw, nullptr, out,
                                                                      static_cast<const uint8_t*>(params), g, heads,
                                                                      nullptr, mask);
    return check_launch("window_attention_forward");
}

}  // extern "C"
