// Masked MS-SSIM on the device (SURVEY.md section 8f, rank 4: the evaluation metric of the RGBA codec).
// Reference semantics: metrics/masked_ms_ssim_torch.py:27-55 (separable valid-mode Gaussian, 11 taps, sigma 1.5, rows then
// columns), :58-121 (_ssim: SSIM / CS maps averaged over the positions where the nearest-resized mask is non-zero),
// :181-265 (ms_ssim: five levels; at each level the mask is binarised and multiplied into both images, then images and
// mask are 2x2 average-pooled with padding = size % 2).  The reference runs ~40 torch kernels per level (five grouped
// convolution pairs, elementwise maps, boolean reductions, three poolings); here a level is TWO launches:
//   ms_ssim_level : one CTA per 16 x 32 tile of the valid region of one (image, channel) plane: the masked X, Y tile with
//                   its 10-pixel apron goes to shared memory once, the five moments are blurred along H into shared
//                   memory, then along W in registers, maps and masked sums follow in the same thread; one atomicAdd pair
//                   per CTA.  HBM traffic = the two planes + the mask, once.
//   ms_ssim_pool  : (X * m, Y * m, m) -> 2x2 average pools of all three in one pass.
// fp32 like the reference; the sums are accumulated in a different order, so values agree to ~1e-6, not bit for bit.
//   ms_ssim_level_bwd : the adjoint of one level (and of the pool that fed the next one), one launch per level from the
//                   coarsest to the finest; see ms_ssim_level_bwd_kernel.  It shares the Gaussian taps (gauss_taps) and
//                   the counted-position rule (counted) with ms_ssim_level, so it weights exactly the positions `counts`
//                   counted.
#include "common.cuh"
#include "status.cuh"

namespace b200 {
namespace {

constexpr int kWin = 11, kApron = kWin - 1;
constexpr int kTH = 16, kTW = 32;                 // output tile (valid-region positions)
constexpr int kIH = kTH + kApron, kIW = kTW + kApron;

struct Gauss {
    float w[kWin];
};

// metrics/masked_ms_ssim_torch.py:13-24 (_fspecial_gauss_1d) in fp32; symmetric bit for bit (w[i] == w[10 - i])
Gauss gauss_taps() {
    Gauss g;
    float s = 0.f;
    for (int i = 0; i < kWin; ++i) {
        const float c = float(i - kWin / 2);
        g.w[i] = expf(-(c * c) / (2.f * 1.5f * 1.5f));
        s += g.w[i];
    }
    for (int i = 0; i < kWin; ++i) g.w[i] /= s;
    return g;
}

// per-level constants: SSIM's C1, C2 and the nearest-resize ratios of the valid region
struct Level {
    float C1, C2, scale_h, scale_w;
};

Level level_consts(int H, int W, float data_range) {
    const int oh = H - kApron, ow = W - kApron;
    return {(0.01f * data_range) * (0.01f * data_range), (0.03f * data_range) * (0.03f * data_range),
            float(double(H) / oh), float(double(W) / ow)};
}

// n_p: whether valid-region position (yy, xx) is averaged: the nearest-resized mask of the valid region (:104-108),
// source index floor(dst * in / out)
__device__ __forceinline__ bool counted(const float* mp, int yy, int xx, int H, int W, float scale_h, float scale_w) {
    const int my = min(int(floorf(float(yy) * scale_h)), H - 1), mx = min(int(floorf(float(xx) * scale_w)), W - 1);
    return mp[int64_t(my) * W + mx] > 0.f;
}

__global__ void __launch_bounds__(256)
ms_ssim_level_kernel(const float* __restrict__ X, const float* __restrict__ Y, const float* __restrict__ mask, int C, int H,
                     int W, float C1, float C2, float scale_h, float scale_w, Gauss g, float* __restrict__ sums,
                     float* __restrict__ counts) {
    __shared__ float sx[kIH][kIW + 1], sy[kIH][kIW + 1];
    __shared__ float v[5][kTH][kIW + 1];           // moments after the blur along H: x, y, xx, yy, xy
    __shared__ float red[3][8];
    const int oh = H - kApron, ow = W - kApron;
    const int tiles_x = (ow + kTW - 1) / kTW;
    const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
    const int c = blockIdx.y, b = blockIdx.z;
    const int y0 = ty * kTH, x0 = tx * kTW;
    const float* xp = X + (int64_t(b) * C + c) * H * W;
    const float* yp = Y + (int64_t(b) * C + c) * H * W;
    const float* mp = mask + int64_t(b) * H * W;
    for (int i = threadIdx.x; i < kIH * kIW; i += 256) {
        const int r = i / kIW, q = i % kIW, yy = y0 + r, xx = x0 + q;
        float a = 0.f, d = 0.f;
        if (yy < H && xx < W) {
            const float m = mp[int64_t(yy) * W + xx] > 0.f ? 1.f : 0.f;        // (mask > 0) multiplied into both images (:236-238)
            a = xp[int64_t(yy) * W + xx] * m;
            d = yp[int64_t(yy) * W + xx] * m;
        }
        sx[r][q] = a;
        sy[r][q] = d;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kTH * kIW; i += 256) {
        const int r = i / kIW, q = i % kIW;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, a4 = 0.f;
#pragma unroll
        for (int k = 0; k < kWin; ++k) {
            const float a = sx[r + k][q], d = sy[r + k][q], w = g.w[k];
            a0 = fmaf(w, a, a0);
            a1 = fmaf(w, d, a1);
            a2 = fmaf(w, a * a, a2);
            a3 = fmaf(w, d * d, a3);
            a4 = fmaf(w, a * d, a4);
        }
        v[0][r][q] = a0; v[1][r][q] = a1; v[2][r][q] = a2; v[3][r][q] = a3; v[4][r][q] = a4;
    }
    __syncthreads();
    float s_ssim = 0.f, s_cs = 0.f, s_n = 0.f;
    for (int i = threadIdx.x; i < kTH * kTW; i += 256) {
        const int r = i / kTW, q = i % kTW, yy = y0 + r, xx = x0 + q;
        if (yy < oh && xx < ow) {
            float m[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int k = 0; k < kWin; ++k) {
                const float w = g.w[k];
#pragma unroll
                for (int f = 0; f < 5; ++f) m[f] = fmaf(w, v[f][r][q + k], m[f]);
            }
            const float mu1 = m[0], mu2 = m[1];
            const float s1 = m[2] - mu1 * mu1, s2 = m[3] - mu2 * mu2, s12 = m[4] - mu1 * mu2;
            const float cs = (2.f * s12 + C2) / (s1 + s2 + C2);
            const float ss = ((2.f * mu1 * mu2 + C1) / (mu1 * mu1 + mu2 * mu2 + C1)) * cs;
            if (counted(mp, yy, xx, H, W, scale_h, scale_w)) {
                s_ssim += ss;
                s_cs += cs;
                s_n += 1.f;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s_ssim += __shfl_xor_sync(0xffffffffu, s_ssim, o);
        s_cs += __shfl_xor_sync(0xffffffffu, s_cs, o);
        s_n += __shfl_xor_sync(0xffffffffu, s_n, o);
    }
    if ((threadIdx.x & 31) == 0) {
        red[0][threadIdx.x >> 5] = s_ssim;
        red[1][threadIdx.x >> 5] = s_cs;
        red[2][threadIdx.x >> 5] = s_n;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, d = 0.f, n = 0.f;
        for (int i = 0; i < 8; ++i) {
            a += red[0][i];
            d += red[1][i];
            n += red[2][i];
        }
        atomicAdd(sums + (int64_t(b) * C + c) * 2, a);
        atomicAdd(sums + (int64_t(b) * C + c) * 2 + 1, d);
        if (c == 0) atomicAdd(counts + b, n);
    }
}

// out sizes: Hp = (H + 2 ph - 2) / 2 + 1 with ph = H % 2 (F.avg_pool2d(kernel 2, padding = size % 2), count_include_pad)
__global__ void __launch_bounds__(256)
ms_ssim_pool_kernel(const float* __restrict__ X, const float* __restrict__ Y, const float* __restrict__ mask, int C, int H,
                    int W, int Hp, int Wp, float* __restrict__ Xo, float* __restrict__ Yo, float* __restrict__ Mo, int64_t n) {
    const int ph = H % 2, pw = W % 2;
    for (int64_t i = blockIdx.x * int64_t(256) + threadIdx.x; i < n; i += int64_t(gridDim.x) * 256) {
        const int xo = int(i % Wp), yo = int((i / Wp) % Hp), b = int(i / (int64_t(Wp) * Hp));
        float mv[4], ms = 0.f;
        int64_t off[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int yy = 2 * yo - ph + (t >> 1), xx = 2 * xo - pw + (t & 1);
            const bool in = yy >= 0 && yy < H && xx >= 0 && xx < W;
            off[t] = in ? int64_t(yy) * W + xx : -1;
            mv[t] = in && mask[int64_t(b) * H * W + off[t]] > 0.f ? 1.f : 0.f;
            ms += mv[t];
        }
        Mo[i] = ms * 0.25f;
        for (int c = 0; c < C; ++c) {
            const float* xp = X + (int64_t(b) * C + c) * H * W;
            const float* yp = Y + (int64_t(b) * C + c) * H * W;
            float a = 0.f, d = 0.f;
#pragma unroll
            for (int t = 0; t < 4; ++t)
                if (off[t] >= 0) {
                    a += xp[off[t]] * mv[t];
                    d += yp[off[t]] * mv[t];
                }
            const int64_t o = ((int64_t(b) * C + c) * Hp + yo) * Wp + xo;
            Xo[o] = a * 0.25f;
            Yo[o] = d * 0.25f;
        }
    }
}

// Backward of one level.  With Xm = X b, Ym = Y b (b = mask > 0), the valid blur G and, per valid position p, the maps of
// the forward (mu1, mu2, s1, s2, s12, B1 = mu1^2 + mu2^2 + C1, B2 = s1 + s2 + C2, l = (2 mu1 mu2 + C1) / B1,
// cs = (2 s12 + C2) / B2), the weight w_p = n_p / N_b of S[b,c] = sum_p w_p l_p cs_p and CS[b,c] = sum_p w_p cs_p gives
//   g_cs = dS w l + dCS w,  g_l = dS w cs,  gE11 = gE22 = -g_cs cs / B2,  gE12 = 2 g_cs / B2,
//   gmu1 = 2 g_l (mu2 - l mu1) / B1 - 2 mu1 gE11 - mu2 gE12     (gmu2: 1 <-> 2)
//   dX = b (G^T gmu1 + 2 Xm G^T gE11 + Ym G^T gE12 + 0.25 dXc[parent])     (dY: X <-> Y, gmu1 -> gmu2)
// G^T, the adjoint of the valid blur, is the full-size correlation with the same (symmetric) taps.  The pool term is the
// adjoint of ms_ssim_pool: every pixel of a 2x2 cell gets a quarter of the gradient of its pooled value.
// One CTA owns a kTH x kTW tile of one (image, channel) plane and writes each of its pixels once (no atomics: the result
// does not depend on scheduling).  The moments are recomputed for the kFH x kFW valid positions whose window touches the
// tile, from the masked X, Y staged with a 10-pixel apron on every side.
constexpr int kBH = kTH + 2 * kApron, kBW = kTW + 2 * kApron, kBP = kBW + 1;   // staged input 36 x 52
constexpr int kFH = kTH + kApron, kFW = kTW + kApron, kFP = kFW + 1;            // gradient fields 26 x 42
constexpr int kBwdSmemFloats = 2 * kBH * kBP + 5 * kFH * kBP + 4 * kFH * kFP;
static_assert(4 * kTH * kFP <= 5 * kFH * kBP, "the transposed H blur reuses the moment buffer");

template <bool DX, bool DY>
__global__ void __launch_bounds__(256)
ms_ssim_level_bwd_kernel(const float* __restrict__ X, const float* __restrict__ Y, const float* __restrict__ mask, int C,
                         int H, int W, Level k, Gauss g, const float* __restrict__ grad, const float* __restrict__ counts,
                         const float* __restrict__ dXc, const float* __restrict__ dYc, float* __restrict__ dX,
                         float* __restrict__ dY) {
    extern __shared__ float smem[];
    float(*sx)[kBP] = reinterpret_cast<float(*)[kBP]>(smem);
    float(*sy)[kBP] = reinterpret_cast<float(*)[kBP]>(smem + kBH * kBP);
    float(*v)[kFH][kBP] = reinterpret_cast<float(*)[kFH][kBP]>(smem + 2 * kBH * kBP);              // moments after the H blur
    float(*f)[kFH][kFP] = reinterpret_cast<float(*)[kFH][kFP]>(smem + 2 * kBH * kBP + 5 * kFH * kBP);   // gE11 gE12 gmu1 gmu2
    float(*t)[kTH][kFP] = reinterpret_cast<float(*)[kTH][kFP]>(smem + 2 * kBH * kBP);              // fields after G^T along H
    const int oh = H - kApron, ow = W - kApron;
    const int tiles_x = (W + kTW - 1) / kTW;
    const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
    const int c = blockIdx.y, b = blockIdx.z;
    const int y0 = ty * kTH, x0 = tx * kTW;
    const int64_t plane = (int64_t(b) * C + c) * H * W;
    const float* mp = mask + int64_t(b) * H * W;
    for (int i = threadIdx.x; i < kBH * kBW; i += 256) {
        const int r = i / kBW, q = i % kBW, yy = y0 - kApron + r, xx = x0 - kApron + q;
        float a = 0.f, d = 0.f;
        if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
            const int64_t o = int64_t(yy) * W + xx;
            if (mp[o] > 0.f) {
                a = X[plane + o];
                d = Y[plane + o];
            }
        }
        sx[r][q] = a;
        sy[r][q] = d;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kFH * kBW; i += 256) {
        const int r = i / kBW, q = i % kBW;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, a4 = 0.f;
#pragma unroll
        for (int j = 0; j < kWin; ++j) {
            const float a = sx[r + j][q], d = sy[r + j][q], w = g.w[j];
            a0 = fmaf(w, a, a0);
            a1 = fmaf(w, d, a1);
            a2 = fmaf(w, a * a, a2);
            a3 = fmaf(w, d * d, a3);
            a4 = fmaf(w, a * d, a4);
        }
        v[0][r][q] = a0; v[1][r][q] = a1; v[2][r][q] = a2; v[3][r][q] = a3; v[4][r][q] = a4;
    }
    __syncthreads();
    const float nb = counts[b] + 1e-10f;
    const float ws = grad[(int64_t(b) * C + c) * 2] / nb, wc = grad[(int64_t(b) * C + c) * 2 + 1] / nb;
    for (int i = threadIdx.x; i < kFH * kFW; i += 256) {
        const int r = i / kFW, q = i % kFW, yy = y0 - kApron + r, xx = x0 - kApron + q;
        float e11 = 0.f, e12 = 0.f, gm1 = 0.f, gm2 = 0.f;
        if (yy >= 0 && yy < oh && xx >= 0 && xx < ow && counted(mp, yy, xx, H, W, k.scale_h, k.scale_w)) {
            float m[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int j = 0; j < kWin; ++j) {
                const float w = g.w[j];
#pragma unroll
                for (int e = 0; e < 5; ++e) m[e] = fmaf(w, v[e][r][q + j], m[e]);
            }
            const float mu1 = m[0], mu2 = m[1];
            const float s1 = m[2] - mu1 * mu1, s2 = m[3] - mu2 * mu2, s12 = m[4] - mu1 * mu2;
            const float B1 = mu1 * mu1 + mu2 * mu2 + k.C1, B2 = s1 + s2 + k.C2;
            const float l = (2.f * mu1 * mu2 + k.C1) / B1, cs = (2.f * s12 + k.C2) / B2;
            const float g_cs = ws * l + wc, g_l = ws * cs;
            e11 = -g_cs * cs / B2;
            e12 = 2.f * g_cs / B2;
            if (DX) gm1 = 2.f * g_l * (mu2 - l * mu1) / B1 - 2.f * mu1 * e11 - mu2 * e12;
            if (DY) gm2 = 2.f * g_l * (mu1 - l * mu2) / B1 - 2.f * mu2 * e11 - mu1 * e12;
        }
        f[0][r][q] = e11;
        f[1][r][q] = e12;
        if (DX) f[2][r][q] = gm1;
        if (DY) f[3][r][q] = gm2;
    }
    __syncthreads();
    // G^T along H: output row r of the tile gathers the field rows r .. r + 10 (taps mirrored = the same taps)
    for (int i = threadIdx.x; i < kTH * kFW; i += 256) {
        const int r = i / kFW, q = i % kFW;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
        for (int j = 0; j < kWin; ++j) {
            const float w = g.w[j];
            a0 = fmaf(w, f[0][r + j][q], a0);
            a1 = fmaf(w, f[1][r + j][q], a1);
            if (DX) a2 = fmaf(w, f[2][r + j][q], a2);
            if (DY) a3 = fmaf(w, f[3][r + j][q], a3);
        }
        t[0][r][q] = a0;
        t[1][r][q] = a1;
        if (DX) t[2][r][q] = a2;
        if (DY) t[3][r][q] = a3;
    }
    __syncthreads();
    const int Hp = (H + 2 * (H % 2) - 2) / 2 + 1, Wp = (W + 2 * (W % 2) - 2) / 2 + 1;
    for (int i = threadIdx.x; i < kTH * kTW; i += 256) {
        const int r = i / kTW, q = i % kTW, yy = y0 + r, xx = x0 + q;
        if (yy >= H || xx >= W) continue;
        float o11 = 0.f, o12 = 0.f, om1 = 0.f, om2 = 0.f;
#pragma unroll
        for (int j = 0; j < kWin; ++j) {
            const float w = g.w[j];
            o11 = fmaf(w, t[0][r][q + j], o11);
            o12 = fmaf(w, t[1][r][q + j], o12);
            if (DX) om1 = fmaf(w, t[2][r][q + j], om1);
            if (DY) om2 = fmaf(w, t[3][r][q + j], om2);
        }
        const float xm = sx[r + kApron][q + kApron], ym = sy[r + kApron][q + kApron];
        const int64_t o = int64_t(yy) * W + xx;
        const bool in = mp[o] > 0.f;
        const int64_t po = ((int64_t(b) * C + c) * Hp + (yy + H % 2) / 2) * Wp + (xx + W % 2) / 2;   // parent in the pool
        if (DX) {
            float d = om1 + 2.f * xm * o11 + ym * o12;
            if (dXc) d += 0.25f * dXc[po];
            dX[plane + o] = in ? d : 0.f;
        }
        if (DY) {
            float d = om2 + 2.f * ym * o11 + xm * o12;
            if (dYc) d += 0.25f * dYc[po];
            dY[plane + o] = in ? d : 0.f;
        }
    }
}

template <bool DX, bool DY>
int launch_level_bwd(const float* X, const float* Y, const float* mask, int B, int C, int H, int W, float data_range,
                     const float* grad, const float* counts, const float* dXc, const float* dYc, float* dX, float* dY,
                     cudaStream_t st) {
    constexpr int smem = kBwdSmemFloats * int(sizeof(float));
    MWA_TRY_CUDA(cudaFuncSetAttribute(ms_ssim_level_bwd_kernel<DX, DY>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem),
                 "ms_ssim_level_backward(smem)");
    dim3 grid(unsigned(((W + kTW - 1) / kTW) * ((H + kTH - 1) / kTH)), unsigned(C), unsigned(B));
    ms_ssim_level_bwd_kernel<DX, DY><<<grid, 256, smem, st>>>(X, Y, mask, C, H, W, level_consts(H, W, data_range),
                                                             gauss_taps(), grad, counts, dXc, dYc, dX, dY);
    return check_launch("ms_ssim_level_backward");
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" {

int ms_ssim_level_forward(const float* X, const float* Y, const float* mask, int B, int C, int H, int W, float data_range,
                          float* sums, float* counts, void* stream) {
    if (!X || !Y || !mask || !sums || !counts || B < 0 || C <= 0) return MWA_ERR_INVALID;
    if (H < kWin || W < kWin) return MWA_ERR_UNSUPPORTED;      // the reference leaves a short dimension unblurred; not needed above 160 px
    if (B == 0) return MWA_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MWA_TRY_CUDA(cudaMemsetAsync(sums, 0, sizeof(float) * 2 * B * C, st), "ms_ssim_level(memset)");
    MWA_TRY_CUDA(cudaMemsetAsync(counts, 0, sizeof(float) * B, st), "ms_ssim_level(memset)");
    const int oh = H - kApron, ow = W - kApron;
    const Level k = level_consts(H, W, data_range);
    dim3 grid(unsigned(((ow + kTW - 1) / kTW) * ((oh + kTH - 1) / kTH)), unsigned(C), unsigned(B));
    ms_ssim_level_kernel<<<grid, 256, 0, st>>>(X, Y, mask, C, H, W, k.C1, k.C2, k.scale_h, k.scale_w, gauss_taps(), sums,
                                              counts);
    return check_launch("ms_ssim_level_forward");
}

int ms_ssim_pool_forward(const float* X, const float* Y, const float* mask, int B, int C, int H, int W, float* Xo, float* Yo,
                         float* Mo, void* stream) {
    if (!X || !Y || !mask || !Xo || !Yo || !Mo || B < 0 || C <= 0 || H <= 0 || W <= 0) return MWA_ERR_INVALID;
    if (B == 0) return MWA_OK;
    const int Hp = (H + 2 * (H % 2) - 2) / 2 + 1, Wp = (W + 2 * (W % 2) - 2) / 2 + 1;
    const int64_t n = int64_t(B) * Hp * Wp;
    int64_t blocks = (n + 255) / 256;
    if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
    ms_ssim_pool_kernel<<<unsigned(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(X, Y, mask, C, H, W, Hp, Wp, Xo, Yo, Mo, n);
    return check_launch("ms_ssim_pool_forward");
}

int ms_ssim_level_backward(const float* X, const float* Y, const float* mask, int B, int C, int H, int W, float data_range,
                           const float* grad, const float* counts, const float* dXc, const float* dYc, float* dX, float* dY,
                           void* stream) {
    if (!X || !Y || !mask || !grad || !counts || B < 0 || C <= 0) return MWA_ERR_INVALID;
    if (H < kWin || W < kWin) return MWA_ERR_UNSUPPORTED;
    if (B == 0) return MWA_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dX && dY) return launch_level_bwd<true, true>(X, Y, mask, B, C, H, W, data_range, grad, counts, dXc, dYc, dX, dY, st);
    if (dX) return launch_level_bwd<true, false>(X, Y, mask, B, C, H, W, data_range, grad, counts, dXc, dYc, dX, dY, st);
    if (dY) return launch_level_bwd<false, true>(X, Y, mask, B, C, H, W, data_range, grad, counts, dXc, dYc, dX, dY, st);
    return MWA_OK;
}

}  // extern "C"
