// 8- and 16-bit RGBA in and out of the codec (DESIGN.md 4.8): the two HBM passes between interleaved uint8 / uint16
// (B, H, W, 4) images and the fp32 NCHW planes the transforms read and write.  One template per direction over the sample
// type T (uint8_t: full scale 255; uint16_t: full scale 65535).
//
// ingest : T (B, H, W, C), C = 4 (RGBA) or 1 (alpha only, the decoder side) -> fp32 image (B, 3, Hp, Wp) and alpha
//          (B, 1, Hp, Wp), Hp / Wp = H / W rounded up to a multiple of 64.  alpha = a / full, image_c = rgb_c / full where
//          a > 0, else 0 (the premultiplication by the binarised alpha that the model was trained on); both divisions
//          IEEE round-to-nearest, as torch's CPU `t.float() / 255` (a multiply by 1/255 differs on 126 of the 256 values).
//          The bottom / right padding is +0.0 in every plane: transparent pixels.
// egress : fp32 x_hat (B, 3, Hp, Wp) + T alpha (B, H, W) -> T (B, H, W, 4): A = alpha, RGB = rint(clamp(x, 0, 1) * full)
//          (fp32 multiply, round half to even) where alpha > 0, else 0; NaN -> 0.
//
// One thread owns 4 horizontally adjacent pixels: the fp32 planes move as float4 (Wp is a multiple of 64, so a 4-pixel group
// never straddles a row and stays 16-byte aligned).  On the integer side a Word is one RGBA pixel, or 4 alpha samples
// (4 / 8 bytes for 8 / 16 bits): the 4 pixels are read / written as 16-byte words (one for 8 bits, two for 16) and the 4
// alpha samples as one Word where the row layout keeps them aligned, else Word by Word (RGBA) or sample by sample (alpha)
// -- coalesced across the warp either way.
#include "common.cuh"
#include "status.cuh"

namespace b200 {
namespace {

constexpr int kThreads = 256;

__host__ __device__ __forceinline__ bool aligned(const void* p, uintptr_t bytes) {
    return (reinterpret_cast<uintptr_t>(p) & (bytes - 1)) == 0;
}

// the sample type's layout: Word holds one RGBA pixel or 4 alpha samples, kBits per sample, full scale kFull
template <typename T> struct Sample;
template <> struct Sample<uint8_t> {
    using Word = uint32_t;
    static constexpr int kBits = 8;
    static constexpr uint32_t kMask = 0xff;
    static constexpr float kFull = 255.0f;
};
template <> struct Sample<uint16_t> {
    using Word = uint64_t;
    static constexpr int kBits = 16;
    static constexpr uint32_t kMask = 0xffff;
    static constexpr float kFull = 65535.0f;
};

// 4 Words (4 RGBA pixels) from / to a 16-byte aligned address: one 16-byte access for 8 bits, two for 16
__device__ __forceinline__ void load4(const uint32_t* p, uint32_t w[4]) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
    w[0] = v.x, w[1] = v.y, w[2] = v.z, w[3] = v.w;
}
__device__ __forceinline__ void load4(const uint64_t* p, uint64_t w[4]) {
    const ulonglong2 u = __ldg(reinterpret_cast<const ulonglong2*>(p)), v = __ldg(reinterpret_cast<const ulonglong2*>(p) + 1);
    w[0] = u.x, w[1] = u.y, w[2] = v.x, w[3] = v.y;
}
__device__ __forceinline__ void store4(uint32_t* p, const uint32_t w[4]) {
    reinterpret_cast<uint4*>(p)[0] = make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ void store4(uint64_t* p, const uint64_t w[4]) {
    reinterpret_cast<ulonglong2*>(p)[0] = make_ulonglong2(w[0], w[1]);
    reinterpret_cast<ulonglong2*>(p)[1] = make_ulonglong2(w[2], w[3]);
}

template <typename T>
__device__ __forceinline__ float unit(uint32_t v) { return __fdiv_rn(float(v), Sample<T>::kFull); }

template <typename T>
__device__ __forceinline__ uint32_t quantise(float v) {
    return uint32_t(rintf(__fmul_rn(fminf(fmaxf(v, 0.0f), 1.0f), Sample<T>::kFull)));       // fmaxf(NaN, 0) = 0
}

// the 4 alpha samples of the group at x0 (x0 + k < W valid) from p: one Word where the layout allows, else sample by sample
template <typename T>
__device__ __forceinline__ void load_alpha4(const T* p, bool full, int x0, int W, uint32_t a[4]) {
    using S = Sample<T>;
    using Word = typename S::Word;
    if (full && aligned(p, sizeof(Word))) {
        const Word w = __ldg(reinterpret_cast<const Word*>(p));
#pragma unroll
        for (int k = 0; k < 4; ++k) a[k] = uint32_t(w >> (S::kBits * k)) & S::kMask;
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (x0 + k < W) a[k] = __ldg(p + k);
    }
}

// grid-stride over B * Hp * (Wp / 4) groups of the padded planes
template <typename T>
__global__ void __launch_bounds__(kThreads)
rgba_ingest_kernel(const T* __restrict__ src, float* __restrict__ image, float* __restrict__ alpha, int H, int W, int C,
                   int Hp, int Wp, int64_t groups) {
    using S = Sample<T>;
    using Word = typename S::Word;
    const int gw = Wp / 4;
    const int64_t plane = int64_t(Hp) * Wp;
    for (int64_t g = blockIdx.x * int64_t(kThreads) + threadIdx.x; g < groups; g += int64_t(gridDim.x) * kThreads) {
        const int x0 = int(g % gw) * 4;
        const int64_t by = g / gw;                       // b * Hp + y
        const int y = int(by % Hp);
        const int64_t b = by / Hp;
        uint32_t a[4] = {0, 0, 0, 0}, r[4] = {0, 0, 0, 0}, gr[4] = {0, 0, 0, 0}, bl[4] = {0, 0, 0, 0};
        if (y < H && x0 < W) {
            const T* p = src + ((b * H + y) * int64_t(W) + x0) * C;
            const bool full = x0 + 4 <= W;
            if (C == 4) {
                if (full && aligned(p, 16)) {
                    Word w[4];
                    load4(reinterpret_cast<const Word*>(p), w);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        r[k] = uint32_t(w[k]) & S::kMask, gr[k] = uint32_t(w[k] >> S::kBits) & S::kMask,
                        bl[k] = uint32_t(w[k] >> (2 * S::kBits)) & S::kMask, a[k] = uint32_t(w[k] >> (3 * S::kBits));
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (x0 + k < W) {
                            const Word w = __ldg(reinterpret_cast<const Word*>(p) + k);
                            r[k] = uint32_t(w) & S::kMask, gr[k] = uint32_t(w >> S::kBits) & S::kMask,
                            bl[k] = uint32_t(w >> (2 * S::kBits)) & S::kMask, a[k] = uint32_t(w >> (3 * S::kBits));
                        }
                }
            } else {
                load_alpha4(p, full, x0, W, a);
            }
        }
        const int64_t off = b * plane + int64_t(y) * Wp + x0;
        reinterpret_cast<float4*>(alpha + off)[0] =
            make_float4(unit<T>(a[0]), unit<T>(a[1]), unit<T>(a[2]), unit<T>(a[3]));
        if (C == 4) {
            float* ip = image + 2 * b * plane + off;     // image batch stride 3 * plane
            const uint32_t* ch[3] = {r, gr, bl};
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float v[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) v[k] = a[k] ? unit<T>(ch[c][k]) : 0.0f;
                reinterpret_cast<float4*>(ip + c * plane)[0] = make_float4(v[0], v[1], v[2], v[3]);
            }
        }
    }
}

// grid-stride over B * H * ceil(W / 4) groups of the image
template <typename T>
__global__ void __launch_bounds__(kThreads)
rgba_egress_kernel(const float* __restrict__ x_hat, const T* __restrict__ alpha_in, T* __restrict__ dst, int H, int W,
                   int Hp, int Wp, int64_t groups) {
    using S = Sample<T>;
    using Word = typename S::Word;
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
        load_alpha4(alpha_in + pix, full, x0, W, a);
        const float* xp = x_hat + 3 * b * plane + int64_t(y) * Wp + x0;
        Word out[4] = {Word(a[0]) << (3 * S::kBits), Word(a[1]) << (3 * S::kBits), Word(a[2]) << (3 * S::kBits),
                       Word(a[3]) << (3 * S::kBits)};
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(xp + c * plane));
            const float vs[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (a[k]) out[k] |= Word(quantise<T>(vs[k])) << (S::kBits * c);
        }
        T* op = dst + pix * 4;
        if (full && aligned(op, 16)) {
            store4(reinterpret_cast<Word*>(op), out);
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (x0 + k < W) reinterpret_cast<Word*>(op)[k] = out[k];
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

// the shared body of the entry points: status checks, then one launch.  The T buffer must be aligned to a whole Word (RGBA:
// 4 bytes for 8 bits, 8 for 16) or a whole sample (alpha only), the units the kernels fall back to.
template <typename T>
int ingest(const T* src, float* image, float* alpha, int B, int H, int W, int C, void* stream, const char* what) {
    if (!size_ok(B, H, W) || (C != 1 && C != 4)) return MWA_ERR_INVALID;
    if (B == 0) return MWA_OK;
    if (!src || !alpha || (C == 4 && !image)) return MWA_ERR_INVALID;
    if (!aligned(alpha, 16) || (C == 4 && (!aligned(image, 16) || !aligned(src, sizeof(typename Sample<T>::Word)))) ||
        !aligned(src, sizeof(T)))
        return MWA_ERR_ALIGNMENT;
    const int Hp = int(padded64(H)), Wp = int(padded64(W));
    const int64_t groups = int64_t(B) * Hp * (Wp / 4);
    rgba_ingest_kernel<T><<<grid_for(groups), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        src, C == 4 ? image : nullptr, alpha, H, W, C, Hp, Wp, groups);
    return check_launch(what);
}

template <typename T>
int egress(const float* x_hat, const T* alpha_in, T* dst, int B, int H, int W, void* stream, const char* what) {
    if (!size_ok(B, H, W)) return MWA_ERR_INVALID;
    if (B == 0) return MWA_OK;
    if (!x_hat || !alpha_in || !dst) return MWA_ERR_INVALID;
    if (!aligned(x_hat, 16) || !aligned(dst, sizeof(typename Sample<T>::Word)) || !aligned(alpha_in, sizeof(T)))
        return MWA_ERR_ALIGNMENT;
    const int Hp = int(padded64(H)), Wp = int(padded64(W));
    const int64_t groups = int64_t(B) * H * ((W + 3) / 4);
    rgba_egress_kernel<T><<<grid_for(groups), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(x_hat, alpha_in, dst, H, W,
                                                                                                Hp, Wp, groups);
    return check_launch(what);
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" {

int rgba8_ingest(const uint8_t* rgba8, float* image, float* alpha, int B, int H, int W, int C, void* stream) {
    return ingest(rgba8, image, alpha, B, H, W, C, stream, "rgba8_ingest");
}

int rgba8_egress(const float* x_hat, const uint8_t* alpha8, uint8_t* rgba8, int B, int H, int W, void* stream) {
    return egress(x_hat, alpha8, rgba8, B, H, W, stream, "rgba8_egress");
}

int rgba16_ingest(const uint16_t* rgba16, float* image, float* alpha, int B, int H, int W, int C, void* stream) {
    return ingest(rgba16, image, alpha, B, H, W, C, stream, "rgba16_ingest");
}

int rgba16_egress(const float* x_hat, const uint16_t* alpha16, uint16_t* rgba16, int B, int H, int W, void* stream) {
    return egress(x_hat, alpha16, rgba16, B, H, W, stream, "rgba16_egress");
}

}  // extern "C"
