// Range-ANS entropy coder of the codec's bitstream (host code; SURVEY.md section 8f, rank 4).
// Reference call sites: models/AutoEncoderRGB_Journal.py:330-368 (compress: BufferedRansEncoder.encode_with_indexes /
// flush) and :374-403 (decompress: RansDecoder.set_stream / decode_stream).  Those classes live in CompressAI
// (compressai.ans, C++; third-party, absent from the reference tree, version unpinned), so this file restates the
// PUBLISHED scheme they implement -- 64-bit rANS state with 32-bit renormalisation words (F. Giesen's rans64), 16-bit
// quantised CDFs selected per symbol by an index, and a 4-bit "bypass" escape for values outside a CDF's support: the
// escape symbol is the CDF's last entry, followed by the number of 4-bit digits (base-15 continuation) and the digits of
//   raw = -2 v - 1 (v < 0)   |   2 (v - max) (v >= max).
// Symbols are pushed in order and coded in reverse so that the decoder reads them forward.  Parity with CompressAI's own
// byte stream is UNPINNED (nothing to compare against); what is tested is the round trip and the stream length against
// the entropy model's estimate.  The coder is serial by construction (one state per stream) and runs on the host; its core
// (rans.cuh) is shared with the device coder of the lane-interleaved format (rans_dev.cu), whose lanes are streams of
// exactly this kind.
#include <cstdint>
#include <cstring>
#include <vector>
#include "rans.cuh"
#include "status.cuh"

using namespace b200;

namespace {
struct VectorEmit {
    std::vector<uint32_t>& words;
    bool operator()(uint32_t w) {
        words.push_back(w);
        return true;
    }
};
}  // namespace

extern "C" {

// cdfs: (ncdf, cdf_stride) int32, row i holds cdf_sizes[i] increasing entries in [0, 2^16]; the support of row i is
// cdf_sizes[i] - 2 regular values + the escape.  Returns the number of BYTES written (a multiple of 4), or a negative status.
MWA_API int64_t rans_encode_with_indexes(const int32_t* symbols, const int32_t* indexes, int64_t n, const int32_t* cdfs, int cdf_stride,
                                 const int32_t* cdf_sizes, const int32_t* offsets, int ncdf, uint8_t* out, int64_t out_capacity) {
    if (n < 0 || (n > 0 && (!symbols || !indexes)) || !cdfs || !cdf_sizes || !offsets || !out || ncdf <= 0) return MWA_ERR_INVALID;
    // validate and code in one backward pass (the coder runs in reverse; an error discards the partial result)
    std::vector<uint32_t> words;
    words.reserve(size_t(n) / 2 + 4);
    VectorEmit emit{words};
    uint64_t x = rans::kRansL;
    for (int64_t i = n; i-- > 0;) {
        const int idx = indexes[i];
        if (idx < 0 || idx >= ncdf || cdf_sizes[idx] > cdf_stride) return MWA_ERR_INVALID;
        if (rans::encode_element_reversed(x, emit, symbols[i], cdfs + int64_t(idx) * cdf_stride, cdf_sizes[idx],
                                          offsets[idx]) != rans::kOk)
            return MWA_ERR_INVALID;
    }
    words.push_back(uint32_t(x >> 32));
    words.push_back(uint32_t(x));
    const int64_t nbytes = int64_t(words.size()) * 4;
    if (nbytes > out_capacity) return MWA_ERR_WORKSPACE;
    // the decoder reads forward: last word written first
    uint32_t* o = reinterpret_cast<uint32_t*>(out);
    for (size_t k = 0; k < words.size(); ++k) {
        const uint32_t w = words[words.size() - 1 - k];
        memcpy(o + k, &w, 4);
    }
    return nbytes;
}

// `state` carries the decoder across calls on one stream (decompress decodes slice by slice): 4 x int64, zero-initialised
// by the caller before the first call.  Returns 0 or a negative status (MWA_ERR_INVALID on a truncated / corrupt stream).
MWA_API int rans_decode_with_indexes(const uint8_t* stream, int64_t nbytes, int64_t* state, const int32_t* indexes, int64_t n,
                             const int32_t* cdfs, int cdf_stride, const int32_t* cdf_sizes, const int32_t* offsets, int ncdf,
                             int32_t* symbols_out) {
    if (!stream || !state || n < 0 || (n > 0 && (!indexes || !symbols_out)) || !cdfs || !cdf_sizes || !offsets || nbytes % 4 != 0)
        return MWA_ERR_INVALID;
    const uint32_t* w = reinterpret_cast<const uint32_t*>(stream);
    rans::Decoder d;
    if (state[0] == 0) {
        d.init(w, 0, nbytes / 4);
    } else {
        d.w = w;
        d.p = state[1];
        d.end = nbytes / 4;
        d.x = uint64_t(state[2]);
        d.ok = true;
    }
    if (!d.ok) return MWA_ERR_INVALID;
    for (int64_t i = 0; i < n; ++i) {
        const int idx = indexes[i];
        if (idx < 0 || idx >= ncdf) return MWA_ERR_INVALID;
        if (!rans::decode_element(d, cdfs + int64_t(idx) * cdf_stride, cdf_sizes[idx], offsets[idx], symbols_out[i]))
            return MWA_ERR_INVALID;
    }
    state[0] = 1;
    state[1] = d.p;
    state[2] = int64_t(d.x);
    return MWA_OK;
}

}  // extern "C"
