// Lane-interleaved rANS on the device: the codec's bitstream coded by one GPU thread per (stream, lane).
// A stream's message is split across L lanes, element g going to lane g mod L; each lane is an ordinary stream of the host
// coder (rans.cu; the core is rans.cuh), so the host coder defines every lane byte for byte.  Stream layout, little-endian
// u32 words: magic, 0x80000000 | version, L, the L lane byte lengths, then the L lane segments in order.
//   encode : walks its lane's elements backwards and writes its segment top-down into a fixed-capacity slot;
//   pack   : one block computes every stream's header and segment offsets, then one block per lane copies its segment, so
//            that all streams of a call end up in one contiguous buffer;
//   decode : decodes elements [position, position + n) of every stream, resuming from the lane states of the last call.
// Nothing here synchronises or allocates; failures are reported in device memory (per lane, per stream).
#include <cub/block/block_scan.cuh>
#include "rans.cuh"
#include "status.cuh"

namespace b200 {
namespace {

constexpr int kLaneThreads = 32;      // one warp per block: the few hundred lane threads of a batch spread over many SMs
constexpr int kPackThreads = 256;

// writes a lane's words top-down into its slot, refusing to pass the slot's bottom
struct SlotEmit {
    uint32_t* top;
    int64_t room;
    __device__ bool operator()(uint32_t w) {
        if (room == 0) return false;
        *--top = w;
        --room;
        return true;
    }
};

__global__ void __launch_bounds__(kLaneThreads) rans_lanes_encode_kernel(
        const int32_t* __restrict__ symbols, const int32_t* __restrict__ indexes, int n_streams, int64_t n, int lanes,
        const int32_t* __restrict__ cdfs, int cdf_stride, const int32_t* __restrict__ cdf_sizes,
        const int32_t* __restrict__ offsets, int ncdf, uint32_t* __restrict__ slots, int64_t slot_words,
        int32_t* __restrict__ lane_words) {
    const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= int64_t(n_streams) * lanes) return;
    const int64_t s = t / lanes, l = t % lanes;
    const int32_t* sym = symbols + s * n;
    const int32_t* idx = indexes + s * n;
    uint32_t* slot_end = slots + (t + 1) * slot_words;
    SlotEmit emit{slot_end, slot_words - 2};                    // two words stay free for the final state
    uint64_t x = rans::kRansL;
    int status = rans::kOk;
    if (l < n) {
        int64_t g = l + (n - 1 - l) / lanes * lanes;
        int32_t i = __ldg(idx + g), v = __ldg(sym + g);
        for (;;) {
            // the next element's symbol and index are loaded while this one is coded (the loop is latency-bound)
            const int64_t next = g - lanes;
            int32_t next_i = 0, next_v = 0;
            if (next >= 0) {
                next_i = __ldg(idx + next);
                next_v = __ldg(sym + next);
            }
            if (i < 0 || i >= ncdf || __ldg(cdf_sizes + i) > cdf_stride) {
                status = rans::kInvalid;
                break;
            }
            status = rans::encode_element_reversed(x, emit, v, cdfs + int64_t(i) * cdf_stride, __ldg(cdf_sizes + i),
                                                   __ldg(offsets + i));
            if (status != rans::kOk || next < 0) break;
            g = next; i = next_i; v = next_v;
        }
    }
    if (status != rans::kOk) {
        lane_words[t] = status == rans::kFull ? MWA_ERR_WORKSPACE : MWA_ERR_INVALID;
        return;
    }
    *--emit.top = uint32_t(x >> 32);
    *--emit.top = uint32_t(x);
    lane_words[t] = int32_t(slot_end - emit.top);
}

// single block: headers, lane destinations (word offsets into `out`) and byte lengths, stream after stream
__global__ void __launch_bounds__(kPackThreads) rans_lanes_offsets_kernel(
        const int32_t* __restrict__ lane_words, int n_streams, int lanes, int64_t* __restrict__ lane_dst,
        int64_t* __restrict__ stream_bytes, uint32_t* __restrict__ out, int64_t out_words) {
    using Scan = cub::BlockScan<int64_t, kPackThreads>;
    __shared__ typename Scan::TempStorage tmp;
    __shared__ int64_t carry;
    __shared__ int failed;                                       // bit 0: an invalid element, bit 1: a full slot
    if (threadIdx.x == 0) failed = 0;
    int64_t base = 0;
    for (int s = 0; s < n_streams; ++s) {
        const int64_t seg0 = base + 3 + lanes;                  // first word of the stream's lane segments
        if (threadIdx.x == 0) carry = 0;
        __syncthreads();
        for (int c = 0; c < lanes; c += kPackThreads) {
            const int l = c + threadIdx.x;
            int64_t w = 0;
            if (l < lanes) {
                w = lane_words[int64_t(s) * lanes + l];
                if (w < 0) {
                    atomicOr(&failed, w == MWA_ERR_WORKSPACE ? 2 : 1);
                    w = 0;
                }
            }
            int64_t before, chunk;
            Scan(tmp).ExclusiveSum(w, before, chunk);
            if (l < lanes) {
                const int64_t dst = seg0 + carry + before;
                lane_dst[int64_t(s) * lanes + l] = dst;
                if (base + 3 + l < out_words) out[base + 3 + l] = uint32_t(w * 4);
            }
            __syncthreads();
            if (threadIdx.x == 0) carry += chunk;
            __syncthreads();
        }
        if (threadIdx.x == 0 && base + 3 <= out_words) {
            out[base] = MWA_RANS_LANES_MAGIC;
            out[base + 1] = 0x80000000u | MWA_RANS_LANES_VERSION;
            out[base + 2] = uint32_t(lanes);
        }
        const int64_t words = 3 + lanes + carry;
        if (threadIdx.x == 0) stream_bytes[s] = words * 4;
        base += words;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        // an invalid element cannot be fixed by a retry with larger slots: report it ahead of a full slot
        int status = (failed & 1) ? MWA_ERR_INVALID : (failed & 2) ? MWA_ERR_WORKSPACE : MWA_OK;
        if (status == MWA_OK && base > out_words) status = MWA_ERR_WORKSPACE;
        stream_bytes[n_streams] = status == 0 ? base * 4 : status;
    }
}

// one block per lane: its segment from the top of its slot to its place in `out`
__global__ void rans_lanes_copy_kernel(const uint32_t* __restrict__ slots, int64_t slot_words,
                                       const int32_t* __restrict__ lane_words, const int64_t* __restrict__ lane_dst,
                                       const int64_t* __restrict__ total, uint32_t* __restrict__ out) {
    if (*total < 0) return;
    const int64_t t = blockIdx.x;
    const int64_t nw = lane_words[t];
    const uint32_t* src = slots + (t + 1) * slot_words - nw;
    uint32_t* dst = out + lane_dst[t];
    for (int64_t k = threadIdx.x; k < nw; k += blockDim.x) dst[k] = src[k];
}

__global__ void __launch_bounds__(kLaneThreads) rans_lanes_decode_kernel(
        const uint32_t* __restrict__ data, int64_t data_words, int64_t* __restrict__ lane_state, int total_lanes,
        const int32_t* __restrict__ stream_lanes, int n_streams, const int32_t* __restrict__ indexes, int64_t n,
        int64_t position, const int32_t* __restrict__ cdfs, int cdf_stride, const int32_t* __restrict__ cdf_sizes,
        const int32_t* __restrict__ offsets, int ncdf, int32_t* __restrict__ symbols, int32_t* __restrict__ status) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total_lanes) return;
    int64_t* st = lane_state + int64_t(t) * 4;
    const int64_t s = st[3] & 0xffffffff, l = st[3] >> 32;
    if (s < 0 || s >= n_streams) return;                        // not a row the caller prepared
    const int64_t lanes = stream_lanes[s];
    if (status[s] != 0) return;                                 // the stream failed in an earlier call
    rans::Decoder d;
    if (l < 0 || l >= lanes || st[1] < 0 || st[2] > data_words || st[1] > st[2]) {
        d.ok = false;
    } else if (st[0] == 0) {                                    // first call: a live state is >= 2^31, never 0
        d.init(data, st[1], st[2]);
    } else {
        d.w = data; d.p = st[1]; d.end = st[2]; d.x = uint64_t(st[0]); d.ok = true;
    }
    if (d.ok) {
        const int32_t* idx = indexes + s * n;
        int32_t* out = symbols + s * n;
        int64_t k = ((l - position) % lanes + lanes) % lanes;
        int32_t i = k < n ? __ldg(idx + k) : 0;
        while (k < n) {
            const int64_t next = k + lanes;
            const int32_t next_i = next < n ? __ldg(idx + next) : 0;     // in flight while element k is decoded
            if (i < 0 || i >= ncdf || !rans::decode_element(d, cdfs + int64_t(i) * cdf_stride, __ldg(cdf_sizes + i),
                                                            __ldg(offsets + i), out[k])) {
                d.ok = false;
                break;
            }
            k = next; i = next_i;
        }
    }
    if (!d.ok) {
        status[s] = MWA_ERR_INVALID;
        return;
    }
    st[0] = int64_t(d.x);
    st[1] = d.p;
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" {

MWA_API int rans_lanes_encode(const int32_t* symbols, const int32_t* indexes, int n_streams, int64_t n, int lanes,
                              const int32_t* cdfs, int cdf_stride, const int32_t* cdf_sizes, const int32_t* offsets,
                              int ncdf, uint32_t* slots, int64_t slot_words, int32_t* lane_words, void* stream) {
    if (n_streams < 0 || n < 0 || lanes < 1 || slot_words < 2 || ncdf <= 0 || cdf_stride < 2 || !cdfs || !cdf_sizes ||
        !offsets || (n > 0 && (!symbols || !indexes)) || (n_streams > 0 && (!slots || !lane_words)))
        return MWA_ERR_INVALID;
    const int64_t threads = int64_t(n_streams) * lanes;
    if (threads == 0) return MWA_OK;
    if (threads > (int64_t(1) << 31) - kLaneThreads) return MWA_ERR_UNSUPPORTED;
    rans_lanes_encode_kernel<<<unsigned((threads + kLaneThreads - 1) / kLaneThreads), kLaneThreads, 0,
                               (cudaStream_t)stream>>>(symbols, indexes, n_streams, n, lanes, cdfs, cdf_stride, cdf_sizes,
                                                       offsets, ncdf, slots, slot_words, lane_words);
    return check_launch("rans_lanes_encode");
}

MWA_API int rans_lanes_pack(const uint32_t* slots, int64_t slot_words, const int32_t* lane_words, int n_streams, int lanes,
                            int64_t* lane_dst, int64_t* stream_bytes, uint32_t* out, int64_t out_words, void* stream) {
    if (n_streams < 1 || lanes < 1 || slot_words < 2 || out_words < 0 || !slots || !lane_words || !lane_dst ||
        !stream_bytes || !out)
        return MWA_ERR_INVALID;
    const int64_t total_lanes = int64_t(n_streams) * lanes;
    if (total_lanes > (int64_t(1) << 31) - 1) return MWA_ERR_UNSUPPORTED;
    cudaStream_t s = (cudaStream_t)stream;
    rans_lanes_offsets_kernel<<<1, kPackThreads, 0, s>>>(lane_words, n_streams, lanes, lane_dst, stream_bytes, out,
                                                         out_words);
    int st = check_launch("rans_lanes_pack");
    if (st != MWA_OK) return st;
    rans_lanes_copy_kernel<<<unsigned(total_lanes), 256, 0, s>>>(slots, slot_words, lane_words, lane_dst,
                                                                 stream_bytes + n_streams, out);
    return check_launch("rans_lanes_pack");
}

MWA_API int rans_lanes_decode(const uint32_t* data, int64_t data_words, int64_t* lane_state, int total_lanes,
                              const int32_t* stream_lanes, int n_streams, const int32_t* indexes, int64_t n,
                              int64_t position, const int32_t* cdfs, int cdf_stride, const int32_t* cdf_sizes,
                              const int32_t* offsets, int ncdf, int32_t* symbols, int32_t* status, void* stream) {
    if (data_words < 0 || total_lanes < 0 || n_streams < 0 || n < 0 || position < 0 || ncdf <= 0 || cdf_stride < 2 ||
        !cdfs || !cdf_sizes || !offsets || (total_lanes > 0 && (!data || !lane_state || !stream_lanes || !status)) ||
        (n > 0 && n_streams > 0 && (!indexes || !symbols)))
        return MWA_ERR_INVALID;
    if (total_lanes == 0 || n == 0) return MWA_OK;
    rans_lanes_decode_kernel<<<unsigned((total_lanes + kLaneThreads - 1) / kLaneThreads), kLaneThreads, 0,
                               (cudaStream_t)stream>>>(data, data_words, lane_state, total_lanes, stream_lanes, n_streams,
                                                       indexes, n, position, cdfs, cdf_stride, cdf_sizes, offsets, ncdf,
                                                       symbols, status);
    return check_launch("rans_lanes_decode");
}

}  // extern "C"
