// Window geometry, keep flags, kept / dropped window lists, the copy of the dropped windows and the host front end that
// launches them, shared by the kernels that work from an ordered list of kept windows (csrc/mwa_sp.cu: 8x8 windows on
// tcgen05; csrc/mwa_small.cu: 4x4 windows in fp32).
// Reference semantics: layers/masked_win_attention.py:6-47 (partition, keep predicate), :237-249 (dropped windows
// contribute zeros, i.e. the block is the identity there).
#pragma once
#include "common.cuh"
#include "params.cuh"
#include "status.cuh"

namespace b200 {
namespace {

constexpr float kNegMask = -100.0f;                 // layers/masked_win_attention.py:214

struct Geom {
    int B, H, W, shift, nwx, nwy, channels_last;
};

__device__ __forceinline__ void window_coords(const Geom& g, int win, int& b, int& wy, int& wx) {
    b = win / (g.nwy * g.nwx);
    const int r = win - b * g.nwy * g.nwx;
    wy = r / g.nwx;
    wx = r - wy * g.nwx;
}
// token t of window (wy, wx): original (un-shifted) pixel
template <int WS>
__device__ __forceinline__ void token_pixel(const Geom& g, int wy, int wx, int t, int& y, int& x) {
    y = wy * WS + t / WS + g.shift;
    if (y >= g.H) y -= g.H;
    x = wx * WS + t % WS + g.shift;
    if (x >= g.W) x -= g.W;
}

// ------------------------------------------------------------------------------------------------ scan / compaction
// one warp per window: keep flag = (sum of the window's alpha != 0)
template <int WS>
__global__ void __launch_bounds__(256)
mwa_scan_kernel(const float* __restrict__ alpha, Geom g, int nwin, uint8_t* __restrict__ flags) {
    constexpr int NTOK = WS * WS;
    const int win = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (win >= nwin) return;
    int b, wy, wx;
    window_coords(g, win, b, wy, wx);
    float a = 0.f;
    for (int t = lane; t < NTOK; t += 32) {
        int y, xx;
        token_pixel<WS>(g, wy, wx, t, y, xx);
        a += __ldg(alpha + (int64_t(b) * g.H + y) * g.W + xx);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) flags[win] = a != 0.f;
}

struct ListWs {             // workspace layout: counts (kept, dropped), keep flags, kept list, dropped list
    int64_t count, flags, list, dlist, total;
    __host__ __device__ explicit ListWs(int64_t nwin) {
        count = 0;
        flags = 16;
        list = align_up(flags + nwin, 16);
        dlist = align_up(list + 4 * (nwin + 16), 16);
        total = align_up(dlist + 4 * (nwin + 16), 256);
    }
};

// single block: ordered lists of kept and of dropped windows (flags == nullptr: every window kept)
__global__ void __launch_bounds__(1024)
mwa_list_compact_kernel(const uint8_t* __restrict__ flags, int nwin, int32_t* __restrict__ list, int32_t* __restrict__ dlist,
                      int32_t* __restrict__ count) {
    __shared__ int part[1024];
    const int tid = threadIdx.x;
    const int per = (nwin + 1023) / 1024;
    const int beg = min(tid * per, nwin), end = min(beg + per, nwin);
    int n = 0;
    for (int i = beg; i < end; ++i) n += flags ? flags[i] : 1;
    part[tid] = n;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const int v = (tid >= o) ? part[tid - o] : 0;
        __syncthreads();
        part[tid] += v;
        __syncthreads();
    }
    int pos = part[tid] - n, dpos = beg - pos;
    for (int i = beg; i < end; ++i) {
        if (!flags || flags[i]) list[pos++] = i;
        else dlist[dpos++] = i;
    }
    if (tid == 1023) {
        count[0] = part[1023];
        count[1] = nwin - part[1023];
    }
}

// out = x on the dropped windows (the block is the identity there, layers/masked_win_attention.py:249 adds zeros).
// Work item = (SEGMENT of up to 8 horizontally adjacent dropped windows, 4 channels), one warp each: with
// shift = ws / 2 a window row sits at half a row's offset (8x8 windows: 32 bytes at a 16-byte offset, i.e. it straddles
// two 32-byte sectors) -- copied window by window every sector would be fetched and written twice (measured 1.7 TB/s);
// a segment is one contiguous row piece of 4 * WS * len bytes per (channel, row), copied as consecutive vectors.
// Transparent regions of real alpha planes are blobs, so segments are long; they are cut at multiples of 8 windows so
// that a fully transparent row still spreads over many warps.  A dropped window starts a segment if wx % 8 == 0 or its
// left neighbour is kept.
template <int VEC>
struct VecT;
template <>
struct VecT<4> { using type = float4; };
template <>
struct VecT<2> { using type = float2; };

template <int WS, int VEC>
__device__ __forceinline__ void copy_segment(const float* __restrict__ xs, float* __restrict__ os, const Geom& g, int wy, int wx,
                                             int len, int nc, int64_t hw, int lane) {
    using V = typename VecT<VEC>::type;
    constexpr int U = 8;
    // vector positions of a (channel, segment): WS rows x (WS / VEC) * len; the (channel, position) pairs of the item are
    // dealt to the lanes position-fastest (consecutive lanes = consecutive vectors of a row), U independent loads in flight
    // Widen the row piece to whole 32-byte sectors where that stays inside the image row: with shift = ws / 2 a piece
    // starts and ends in the middle of a sector, and a half-written sector costs a read-modify-write.  The extra 16 bytes
    // on either side belong to a neighbouring window: if that one is dropped it receives the same values from its own
    // copy, if it is kept the attention kernel (later in the stream) overwrites every pixel of it.
    int px_start = wx * WS + g.shift, px_end = px_start + WS * len;
    if (VEC == 4 && px_end <= g.W) {
        if (px_start % 8 == 4) px_start -= 4;
        if (px_end % 8 == 4 && px_end + 4 <= g.W) px_end += 4;
    }
    const int per_row = (px_end - px_start) / VEC, npos = WS * per_row, total = npos * nc;
    for (int base = lane; base < total; base += 32 * U) {
        V v[U];
        int64_t off[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int idx = base + 32 * u;
            off[u] = -1;
            if (idx < total) {
                const int c = idx / npos, pos = idx - c * npos;
                const int r = pos / per_row, k = pos - r * per_row;
                int py = wy * WS + r + g.shift, px = px_start + VEC * k;
                if (py >= g.H) py -= g.H;
                if (px >= g.W) px -= g.W;
                off[u] = int64_t(c) * hw + int64_t(py) * g.W + px;
                v[u] = __ldcs(reinterpret_cast<const V*>(xs + off[u]));
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (off[u] >= 0) __stcs(reinterpret_cast<V*>(os + off[u]), v[u]);
    }
}

template <int WS>
__global__ void __launch_bounds__(256)
mwa_copy_dropped_kernel(const float* __restrict__ x, float* __restrict__ out, Geom g, int C,
                        const uint8_t* __restrict__ flags, const int32_t* __restrict__ dlist,
                        const int32_t* __restrict__ count) {
    constexpr int SEG = 8, CPP = 4;                      // channels per work item: many small items, one round each
    const int n = count[1];
    const int lane = threadIdx.x & 31, gw = blockIdx.x * 8 + (threadIdx.x >> 5), nw = gridDim.x * 8;
    const int64_t hw = int64_t(g.H) * g.W;
    const int parts = (C + CPP - 1) / CPP;
    for (int64_t i = gw; i < int64_t(n) * parts; i += nw) {
        const int win = dlist[i / parts];
        int b, wy, wx;
        window_coords(g, win, b, wy, wx);
        if (wx % SEG != 0 && !flags[win - 1]) continue;      // not the head of its segment
        int len = 1;
        while ((wx + len) % SEG != 0 && wx + len < g.nwx && !flags[win + len]) ++len;
        const int c0 = int(i % parts) * CPP;
        const int nc = min(CPP, C - c0);
        if (nc <= 0) continue;
        const float* xs = x + (int64_t(b) * C + c0) * hw;
        float* os = out + (int64_t(b) * C + c0) * hw;
        if (WS % 4 == 0 && g.shift % 4 == 0 && g.W % 4 == 0) {
            copy_segment<WS, 4>(xs, os, g, wy, wx, len, nc, hw, lane);
        } else if (g.shift % 2 == 0 && g.W % 2 == 0) {
            copy_segment<WS, 2>(xs, os, g, wy, wx, len, nc, hw, lane);
        } else {
            for (int t = lane; t < WS * WS * len; t += 32) {
                int py, px;
                token_pixel<WS>(g, wy, wx + t / (WS * WS), t % (WS * WS), py, px);
                const int64_t off = int64_t(py) * g.W + px;
                for (int c = 0; c < nc; ++c) os[off + c * hw] = __ldg(xs + off + c * hw);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ host front end
// Everything a list-based forward does around its main kernel: checks the window count and the workspace, builds the
// keep flags and the ordered kept / dropped lists in the workspace (alpha == nullptr keeps every window), copies the
// dropped windows x -> out, then calls launch(nwin, list, count) for the main kernel (count[0] = kept windows, on the
// device) and finally copies the kept count to kept_count (may be nullptr).
template <int WS, class Launch>
int mwa_forward_lists(const float* x, const float* alpha, float* out, const Geom& geo, int C, int32_t* kept_count,
                      void* workspace, int64_t workspace_bytes, cudaStream_t st, Launch launch) {
    const int64_t nwin64 = int64_t(geo.B) * geo.nwx * geo.nwy;
    if (nwin64 > 0x3fffffffll) return MWA_ERR_UNSUPPORTED;
    const int nwin = static_cast<int>(nwin64);
    const ListWs ws(nwin);
    if (!workspace || workspace_bytes < ws.total) return MWA_ERR_WORKSPACE;
    if (!aligned16(workspace)) return MWA_ERR_ALIGNMENT;
    uint8_t* wsp = static_cast<uint8_t*>(workspace);
    int32_t* count = reinterpret_cast<int32_t*>(wsp + ws.count);
    uint8_t* flags = wsp + ws.flags;
    int32_t* list = reinterpret_cast<int32_t*>(wsp + ws.list);
    int32_t* dlist = reinterpret_cast<int32_t*>(wsp + ws.dlist);
    int rc;
    if (alpha != nullptr) {
        mwa_scan_kernel<WS><<<(nwin + 7) / 8, 256, 0, st>>>(alpha, geo, nwin, flags);
        rc = check_launch("mwa_forward(scan)");
        if (rc != MWA_OK) return rc;
    }
    mwa_list_compact_kernel<<<1, 1024, 0, st>>>(alpha ? flags : nullptr, nwin, list, dlist, count);
    rc = check_launch("mwa_forward(compact)");
    if (rc != MWA_OK) return rc;
    if (alpha != nullptr && out != x) {
        mwa_copy_dropped_kernel<WS><<<kNumSMs * 8, 256, 0, st>>>(x, out, geo, C, flags, dlist, count);
        rc = check_launch("mwa_forward(copy dropped)");
        if (rc != MWA_OK) return rc;
    }
    rc = launch(nwin, list, count);
    if (rc != MWA_OK) return rc;
    if (kept_count)
        MWA_TRY_CUDA(cudaMemcpyAsync(kept_count, count, sizeof(int32_t), cudaMemcpyDeviceToDevice, st), "mwa_forward(kept_count)");
    return MWA_OK;
}

}  // namespace
}  // namespace b200
