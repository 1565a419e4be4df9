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
// Both also run on tiles (rgba*_ingest_tiles / rgba*_egress_tiles): a launch covers tiles [first, first + count) of the
// B * ceil(H / Th) * ceil(W / Tw) tiles of Th x Tw (multiples of 64) of the batch, in the order image, tile row, tile column.
// The ingest writes the planes of those tiles, (count, 3 or 1, Th, Tw), padded with transparent pixels past the image; the
// egress reads (count, 3, Th, Tw) and writes the pixels of the image those tiles cover, and no other byte.  The untiled
// entry points are the case of one Hp x Wp tile per image.
//
// One thread owns 4 horizontally adjacent pixels: the fp32 planes move as float4 (Tw is a multiple of 64, so a 4-pixel group
// never straddles a row or a tile and stays 16-byte aligned).  On the integer side a Word is one RGBA pixel, or 4 alpha samples
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

// The tiles a launch covers: tile n = (b * ty + i) * tx + j (image b, tile row i, tile column j) covers rows
// [i * Th, (i + 1) * Th) and columns [j * Tw, (j + 1) * Tw) of image b; a launch covers tiles [first, first + count), and
// local tile t = n - first owns planes t of (count, C, Th, Tw).  One tile per image (ty = tx = 1; Th = Hp, Tw = Wp for the
// untiled entry points) is launched as images [first, first + count) with kTiled = false: the image-row traversal, whose
// index arithmetic is that of the untiled kernels, so the untiled conversion costs what it cost before tiles existed.
struct Tiles {
    int64_t tx, per_image, first;                    // per_image = ty * tx

    // image b and the image coordinates (y0, x0) of the top left pixel of local tile t
    __device__ __forceinline__ void origin(int64_t t, int Th, int Tw, int64_t& b, int& y0, int& x0) const {
        const int64_t n = first + t;
        b = n / per_image;
        const int64_t r = n - b * per_image, i = r / tx;
        y0 = int(i * Th), x0 = int((r - i * tx) * Tw);
    }
};

// local tile t, tile row yt and tile column xt of group g: 32-bit arithmetic, as a launch has count * Th * Tw / 4 < 2^31 / 192
// groups
__device__ __forceinline__ void split(int64_t g, int Th, int Tw, int64_t& t, int& yt, int& xt) {
    const uint32_t gw = uint32_t(Tw) / 4, row = uint32_t(g) / gw, tt = row / uint32_t(Th);
    xt = int(uint32_t(g) - row * gw) * 4, yt = int(row - tt * uint32_t(Th)), t = tt;
}

// grid-stride over count * Th * (Tw / 4) groups of the tile planes.  kTiled = false: one tile per image, src starting at
// the launch's first image (t = b)
template <typename T, bool kTiled>
__global__ void __launch_bounds__(kThreads)
rgba_ingest_kernel(const T* __restrict__ src, float* __restrict__ image, float* __restrict__ alpha, int H, int W, int C,
                   int Th, int Tw, int64_t groups, Tiles tl) {
    using S = Sample<T>;
    using Word = typename S::Word;
    const int gw = Tw / 4;
    const int64_t plane = int64_t(Th) * Tw;
    for (int64_t g = blockIdx.x * int64_t(kThreads) + threadIdx.x; g < groups; g += int64_t(gridDim.x) * kThreads) {
        int64_t t, b;
        int yt, xt, y, x0;
        if constexpr (kTiled) {
            split(g, Th, Tw, t, yt, xt);
            tl.origin(t, Th, Tw, b, y, x0);
            y += yt, x0 += xt;
        } else {
            xt = int(g % gw) * 4;
            const int64_t by = g / gw;                   // b * Th + y
            yt = int(by % Th);
            t = by / Th;
            b = t, y = yt, x0 = xt;
        }
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
        const int64_t off = t * plane + int64_t(yt) * Tw + xt;
        reinterpret_cast<float4*>(alpha + off)[0] =
            make_float4(unit<T>(a[0]), unit<T>(a[1]), unit<T>(a[2]), unit<T>(a[3]));
        if (C == 4) {
            float* ip = image + 2 * t * plane + off;     // image tile stride 3 * plane
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

// kTiled: grid-stride over count * Th * (Tw / 4) groups of the tile planes, the groups outside the image writing nothing;
// else over count * H * ceil(W / 4) groups of the images (one tile each), alpha_in and dst starting at the launch's first
template <typename T, bool kTiled>
__global__ void __launch_bounds__(kThreads)
rgba_egress_kernel(const float* __restrict__ x_hat, const T* __restrict__ alpha_in, T* __restrict__ dst, int H, int W,
                   int Th, int Tw, int64_t groups, Tiles tl) {
    using S = Sample<T>;
    using Word = typename S::Word;
    const int gw = (W + 3) / 4;
    const int64_t plane = int64_t(Th) * Tw;
    for (int64_t g = blockIdx.x * int64_t(kThreads) + threadIdx.x; g < groups; g += int64_t(gridDim.x) * kThreads) {
        int64_t t, pix;
        int yt, xt, x0;
        if constexpr (kTiled) {
            int64_t b;
            int y;
            split(g, Th, Tw, t, yt, xt);
            tl.origin(t, Th, Tw, b, y, x0);
            y += yt, x0 += xt;
            if (y >= H || x0 >= W) continue;
            pix = (b * H + y) * int64_t(W) + x0;         // first pixel of the group in (B, H, W)
        } else {
            x0 = int(g % gw) * 4;
            const int64_t by = g / gw;                   // b * H + y
            yt = int(by % H), t = by / H, xt = x0;
            pix = by * W + x0;
        }
        const bool full = x0 + 4 <= W;
        uint32_t a[4] = {0, 0, 0, 0};
        load_alpha4(alpha_in + pix, full, x0, W, a);
        const float* xp = x_hat + 3 * t * plane + int64_t(yt) * Tw + xt;
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

constexpr int64_t kLimit = int64_t(1) << 31;

inline int64_t padded64(int n) { return (int64_t(n) + 63) / 64 * 64; }

// B, H, W valid and B * Hp * Wp * 48 (the element count of the forward's largest activation: 192 channels at 1/2 scale)
// below 2^31, the int32 element indexing of the transforms' kernels
bool size_ok(int B, int H, int W) {
    if (B < 0 || H < 1 || W < 1) return false;
    const int64_t hp = padded64(H), wp = padded64(W);
    if (hp >= kLimit || wp >= kLimit || hp * wp >= kLimit) return false;
    return int64_t(B) <= (kLimit - 1) / (hp * wp * 48);
}

// B, H, W valid, Th and Tw positive multiples of 64, tiles [first, first + count) within the B * ceil(H / Th) *
// ceil(W / Tw) tiles of the batch, and for count > 0 count * Th * Tw * 48 below 2^31 (the same bound as size_ok, for one
// call's planes) and ty * Th, tx * Tw below 2^31 (the kernels' int image coordinates)
bool tiles_ok(int B, int H, int W, int Th, int Tw, int64_t first, int count, Tiles& tl) {
    if (B < 0 || H < 1 || W < 1 || Th < 64 || Tw < 64 || Th % 64 || Tw % 64 || first < 0 || count < 0) return false;
    const int64_t ty = (int64_t(H) + Th - 1) / Th, tx = (int64_t(W) + Tw - 1) / Tw;
    if (first > INT64_MAX - count) return false;
    const int64_t end = first + count, per_image = ty * tx;    // ty, tx < 2^25: no overflow
    if (end / per_image + (end % per_image != 0) > B) return false;
    const int64_t tile = int64_t(Th) * Tw;
    // what a launch touches: count * Th * Tw * 48 below 2^31, and tile rows and columns that end within int coordinates
    if (count > 0 && (tile >= kLimit || count > (kLimit - 1) / (tile * 48) || ty * Th >= kLimit || tx * Tw >= kLimit))
        return false;
    tl = Tiles{tx, per_image, first};
    return true;
}

unsigned grid_for(int64_t groups) {
    const int64_t blocks = (groups + kThreads - 1) / kThreads;
    return unsigned(blocks < 65535 * 16 ? blocks : 65535 * 16);      // grid-stride beyond ~268 M groups
}

// the shared bodies of the entry points: status checks, then one launch.  The T buffer must be aligned to a whole Word
// (RGBA: 4 bytes for 8 bits, 8 for 16) or a whole sample (alpha only), the units the kernels fall back to.
template <typename T>
int ingest(const T* src, float* image, float* alpha, int B, int H, int W, int C, int Th, int Tw, int64_t first, int count,
           void* stream, const char* what) {
    Tiles tl;
    if (!tiles_ok(B, H, W, Th, Tw, first, count, tl) || (C != 1 && C != 4)) return MWA_ERR_INVALID;
    if (count == 0) return MWA_OK;
    if (!src || !alpha || (C == 4 && !image)) return MWA_ERR_INVALID;
    if (!aligned(alpha, 16) || (C == 4 && (!aligned(image, 16) || !aligned(src, sizeof(typename Sample<T>::Word)))) ||
        !aligned(src, sizeof(T)))
        return MWA_ERR_ALIGNMENT;
    const int64_t groups = int64_t(count) * Th * (Tw / 4);
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (tl.per_image == 1)
        rgba_ingest_kernel<T, false><<<grid_for(groups), kThreads, 0, s>>>(src + first * H * int64_t(W) * C,
                                                                          C == 4 ? image : nullptr, alpha, H, W, C, Th, Tw,
                                                                          groups, tl);
    else
        rgba_ingest_kernel<T, true><<<grid_for(groups), kThreads, 0, s>>>(src, C == 4 ? image : nullptr, alpha, H, W, C,
                                                                         Th, Tw, groups, tl);
    return check_launch(what);
}

template <typename T>
int egress(const float* x_hat, const T* alpha_in, T* dst, int B, int H, int W, int Th, int Tw, int64_t first, int count,
           void* stream, const char* what) {
    Tiles tl;
    if (!tiles_ok(B, H, W, Th, Tw, first, count, tl)) return MWA_ERR_INVALID;
    if (count == 0) return MWA_OK;
    if (!x_hat || !alpha_in || !dst) return MWA_ERR_INVALID;
    if (!aligned(x_hat, 16) || !aligned(dst, sizeof(typename Sample<T>::Word)) || !aligned(alpha_in, sizeof(T)))
        return MWA_ERR_ALIGNMENT;
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (tl.per_image == 1) {
        const int64_t groups = int64_t(count) * H * ((W + 3) / 4), pix = first * H * int64_t(W);
        rgba_egress_kernel<T, false><<<grid_for(groups), kThreads, 0, s>>>(x_hat, alpha_in + pix, dst + pix * 4, H, W,
                                                                          Th, Tw, groups, tl);
    } else {
        const int64_t groups = int64_t(count) * Th * (Tw / 4);
        rgba_egress_kernel<T, true><<<grid_for(groups), kThreads, 0, s>>>(x_hat, alpha_in, dst, H, W, Th, Tw, groups, tl);
    }
    return check_launch(what);
}

// the untiled entry points: one tile of Hp x Wp per image, behind their own size guard
template <typename T>
int ingest(const T* src, float* image, float* alpha, int B, int H, int W, int C, void* stream, const char* what) {
    if (!size_ok(B, H, W)) return MWA_ERR_INVALID;
    return ingest(src, image, alpha, B, H, W, C, int(padded64(H)), int(padded64(W)), 0, B, stream, what);
}

template <typename T>
int egress(const float* x_hat, const T* alpha_in, T* dst, int B, int H, int W, void* stream, const char* what) {
    if (!size_ok(B, H, W)) return MWA_ERR_INVALID;
    return egress(x_hat, alpha_in, dst, B, H, W, int(padded64(H)), int(padded64(W)), 0, B, stream, what);
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

int rgba8_ingest_tiles(const uint8_t* rgba8, float* image, float* alpha, int B, int H, int W, int C, int Th, int Tw,
                       int64_t first, int count, void* stream) {
    return ingest(rgba8, image, alpha, B, H, W, C, Th, Tw, first, count, stream, "rgba8_ingest_tiles");
}

int rgba8_egress_tiles(const float* x_hat, const uint8_t* alpha8, uint8_t* rgba8, int B, int H, int W, int Th, int Tw,
                       int64_t first, int count, void* stream) {
    return egress(x_hat, alpha8, rgba8, B, H, W, Th, Tw, first, count, stream, "rgba8_egress_tiles");
}

int rgba16_ingest_tiles(const uint16_t* rgba16, float* image, float* alpha, int B, int H, int W, int C, int Th, int Tw,
                        int64_t first, int count, void* stream) {
    return ingest(rgba16, image, alpha, B, H, W, C, Th, Tw, first, count, stream, "rgba16_ingest_tiles");
}

int rgba16_egress_tiles(const float* x_hat, const uint16_t* alpha16, uint16_t* rgba16, int B, int H, int W, int Th, int Tw,
                        int64_t first, int count, void* stream) {
    return egress(x_hat, alpha16, rgba16, B, H, W, Th, Tw, first, count, stream, "rgba16_egress_tiles");
}

}  // extern "C"
