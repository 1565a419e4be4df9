// 8-bit RGBA in and out of the codec (DESIGN.md 4.8): the two HBM passes between interleaved uint8 (B, H, W, 4) images and
// the fp32 NCHW planes the transforms read and write.
//
// ingest : uint8 (B, H, W, C), C = 4 (RGBA) or 1 (alpha only, the decoder side) -> fp32 image (B, 3, Hp, Wp) and alpha
//          (B, 1, Hp, Wp), Hp / Wp = H / W rounded up to a multiple of 64.  alpha = a / 255, image_c = rgb_c / 255 where
//          a > 0, else 0 (the premultiplication by the binarised alpha that the model was trained on); both divisions
//          IEEE round-to-nearest, as torch's CPU `t.float() / 255` (a multiply by 1/255 differs on 126 of the 256 values).
//          The bottom / right padding is +0.0 in every plane: transparent pixels.
// egress : fp32 x_hat (B, 3, Hp, Wp) + uint8 alpha (B, H, W) -> uint8 (B, H, W, 4): A = alpha, RGB = rint(clamp(x, 0, 1) * 255)
//          (fp32 multiply, round half to even) where alpha > 0, else 0; NaN -> 0.
//
// One thread owns 4 horizontally adjacent pixels: the fp32 planes move as float4 (Wp is a multiple of 64, so a 4-pixel group
// never straddles a row and stays 16-byte aligned); the uint8 side is read / written as 16-byte (RGBA) or 4-byte (alpha)
// words where the row layout keeps them aligned, else pixel by pixel -- coalesced across the warp either way.
#include "common.cuh"
#include "status.cuh"

namespace b200 {
namespace {

constexpr int kThreads = 256;

__host__ __device__ __forceinline__ bool aligned(const void* p, uintptr_t bytes) {
    return (reinterpret_cast<uintptr_t>(p) & (bytes - 1)) == 0;
}

__device__ __forceinline__ float unit(uint32_t v) { return __fdiv_rn(float(v), 255.0f); }

__device__ __forceinline__ uint32_t quantise(float v) {
    return uint32_t(rintf(__fmul_rn(fminf(fmaxf(v, 0.0f), 1.0f), 255.0f)));       // fmaxf(NaN, 0) = 0
}

// grid-stride over B * Hp * (Wp / 4) groups of the padded planes
__global__ void __launch_bounds__(kThreads)
rgba8_ingest_kernel(const uint8_t* __restrict__ src, float* __restrict__ image, float* __restrict__ alpha, int H, int W,
                    int C, int Hp, int Wp, int64_t groups) {
    const int gw = Wp / 4;
    const int64_t plane = int64_t(Hp) * Wp;
    for (int64_t g = blockIdx.x * int64_t(kThreads) + threadIdx.x; g < groups; g += int64_t(gridDim.x) * kThreads) {
        const int x0 = int(g % gw) * 4;
        const int64_t by = g / gw;                       // b * Hp + y
        const int y = int(by % Hp);
        const int64_t b = by / Hp;
        uint32_t a[4] = {0, 0, 0, 0}, r[4] = {0, 0, 0, 0}, gr[4] = {0, 0, 0, 0}, bl[4] = {0, 0, 0, 0};
        if (y < H && x0 < W) {
            const uint8_t* p = src + ((b * H + y) * int64_t(W) + x0) * C;
            const bool full = x0 + 4 <= W;
            if (C == 4) {
                if (full && aligned(p, 16)) {
                    const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
                    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        r[k] = w[k] & 0xff, gr[k] = (w[k] >> 8) & 0xff, bl[k] = (w[k] >> 16) & 0xff, a[k] = w[k] >> 24;
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (x0 + k < W) {
                            const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(p) + k);
                            r[k] = w & 0xff, gr[k] = (w >> 8) & 0xff, bl[k] = (w >> 16) & 0xff, a[k] = w >> 24;
                        }
                }
            } else if (full && aligned(p, 4)) {
                const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(p));
#pragma unroll
                for (int k = 0; k < 4; ++k) a[k] = (w >> (8 * k)) & 0xff;
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (x0 + k < W) a[k] = __ldg(p + k);
            }
        }
        const int64_t off = b * plane + int64_t(y) * Wp + x0;
        reinterpret_cast<float4*>(alpha + off)[0] = make_float4(unit(a[0]), unit(a[1]), unit(a[2]), unit(a[3]));
        if (C == 4) {
            float* ip = image + 2 * b * plane + off;     // image batch stride 3 * plane
            const uint32_t* ch[3] = {r, gr, bl};
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float v[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) v[k] = a[k] ? unit(ch[c][k]) : 0.0f;
                reinterpret_cast<float4*>(ip + c * plane)[0] = make_float4(v[0], v[1], v[2], v[3]);
            }
        }
    }
}

// grid-stride over B * H * ceil(W / 4) groups of the image
__global__ void __launch_bounds__(kThreads)
rgba8_egress_kernel(const float* __restrict__ x_hat, const uint8_t* __restrict__ alpha8, uint8_t* __restrict__ dst, int H,
                    int W, int Hp, int Wp, int64_t groups) {
    const int gw = (W + 3) / 4;
    const int64_t plane = int64_t(Hp) * Wp;
    for (int64_t g = blockIdx.x * int64_t(kThreads) + threadIdx.x; g < groups; g += int64_t(gridDim.x) * kThreads) {
        const int x0 = int(g % gw) * 4;
        const int64_t by = g / gw;                       // b * H + y
        const int y = int(by % H);
        const int64_t b = by / H;
        const int64_t pix = by * W + x0;                 // first pixel of the group in (B, H, W)
        const bool full = x0 + 4 <= W;
        uint32_t a[4] = {0, 0, 0, 0};
        const uint8_t* ap = alpha8 + pix;
        if (full && aligned(ap, 4)) {
            const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(ap));
#pragma unroll
            for (int k = 0; k < 4; ++k) a[k] = (w >> (8 * k)) & 0xff;
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (x0 + k < W) a[k] = __ldg(ap + k);
        }
        const float* xp = x_hat + 3 * b * plane + int64_t(y) * Wp + x0;
        uint32_t out[4] = {a[0] << 24, a[1] << 24, a[2] << 24, a[3] << 24};
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(xp + c * plane));
            const float vs[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (a[k]) out[k] |= quantise(vs[k]) << (8 * c);
        }
        uint8_t* op = dst + pix * 4;
        if (full && aligned(op, 16)) {
            reinterpret_cast<uint4*>(op)[0] = make_uint4(out[0], out[1], out[2], out[3]);
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (x0 + k < W) reinterpret_cast<uint32_t*>(op)[k] = out[k];
        }
    }
}

inline int64_t padded64(int n) { return (int64_t(n) + 63) / 64 * 64; }

// B, H, W valid and B * Hp * Wp * 48 (the element count of the forward's largest activation: 192 channels at 1/2 scale)
// below 2^31, the int32 element indexing of the transforms' kernels
bool size_ok(int B, int H, int W) {
    if (B < 0 || H < 1 || W < 1) return false;
    const int64_t limit = int64_t(1) << 31;
    const int64_t hp = padded64(H), wp = padded64(W);
    if (hp >= limit || wp >= limit || hp * wp >= limit) return false;
    return int64_t(B) <= (limit - 1) / (hp * wp * 48);
}

unsigned grid_for(int64_t groups) {
    const int64_t blocks = (groups + kThreads - 1) / kThreads;
    return unsigned(blocks < 65535 * 16 ? blocks : 65535 * 16);      // grid-stride beyond ~268 M groups
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" {

int rgba8_ingest(const uint8_t* rgba8, float* image, float* alpha, int B, int H, int W, int C, void* stream) {
    if (!size_ok(B, H, W) || (C != 1 && C != 4)) return MWA_ERR_INVALID;
    if (B == 0) return MWA_OK;
    if (!rgba8 || !alpha || (C == 4 && !image)) return MWA_ERR_INVALID;
    if (!aligned(alpha, 16) || (C == 4 && (!aligned(image, 16) || !aligned(rgba8, 4)))) return MWA_ERR_ALIGNMENT;
    const int Hp = int(padded64(H)), Wp = int(padded64(W));
    const int64_t groups = int64_t(B) * Hp * (Wp / 4);
    rgba8_ingest_kernel<<<grid_for(groups), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        rgba8, C == 4 ? image : nullptr, alpha, H, W, C, Hp, Wp, groups);
    return check_launch("rgba8_ingest");
}

int rgba8_egress(const float* x_hat, const uint8_t* alpha8, uint8_t* rgba8, int B, int H, int W, void* stream) {
    if (!size_ok(B, H, W)) return MWA_ERR_INVALID;
    if (B == 0) return MWA_OK;
    if (!x_hat || !alpha8 || !rgba8) return MWA_ERR_INVALID;
    if (!aligned(x_hat, 16) || !aligned(rgba8, 4)) return MWA_ERR_ALIGNMENT;
    const int Hp = int(padded64(H)), Wp = int(padded64(W));
    const int64_t groups = int64_t(B) * H * ((W + 3) / 4);
    rgba8_egress_kernel<<<grid_for(groups), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(x_hat, alpha8, rgba8, H, W,
                                                                                              Hp, Wp, groups);
    return check_launch("rgba8_egress");
}

}  // extern "C"
