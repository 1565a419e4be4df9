// Core of the range-ANS coder (csrc/rans.cu), shared by the host coder and the lane-interleaved device coder
// (csrc/rans_dev.cu): state update, renormalisation, 4-bit bypass digits and the escape expansion of one symbol.
// 64-bit state, 32-bit renormalisation words (F. Giesen's rans64), 16-bit quantised CDFs.  A value outside a CDF's support
// is coded as the escape symbol (the CDF's last interval), then the number of 4-bit digits (base-15 continuation: digits
// of 15 followed by a remainder < 15), then the digits, low first, of
//   raw = -2 v - 1 (v < 0)   |   2 (v - max) (v >= max).
// The message is coded in reverse so that the decoder reads it forward: encode_element_reversed() emits one element's
// pieces in the reverse of the order decode_element() reads them.
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define RANS_HD __host__ __device__ __forceinline__
// the word sink of the host coder is host code; these templates only ever run it from host instantiations
#define RANS_HD_TEMPLATE _Pragma("nv_exec_check_disable")
#else
#define RANS_HD_TEMPLATE
#define RANS_HD inline
#endif

namespace b200 {
namespace rans {

constexpr int kPrecision = 16, kBypassPrecision = 4, kMaxBypass = (1 << kBypassPrecision) - 1;
constexpr int kMaxDigits = 8;                          // raw is a uint32: at most 8 digits of 4 bits
constexpr uint64_t kRansL = uint64_t(1) << 31;          // lower bound of the normalisation interval

// outcome of encoding one element
enum { kOk = 0, kInvalid = 1, kFull = 2 };

// `emit(word)` appends one renormalisation word and returns false when there is no room left
RANS_HD_TEMPLATE
template <class Emit>
RANS_HD bool enc_put(uint64_t& x, Emit& emit, uint32_t start, uint32_t freq) {
    const uint64_t x_max = ((kRansL >> kPrecision) << 32) * freq;
    if (x >= x_max) {
        if (!emit(uint32_t(x))) return false;
        x >>= 32;
    }
    x = ((x / freq) << kPrecision) + (x % freq) + start;
    return true;
}

RANS_HD_TEMPLATE
template <class Emit>
RANS_HD bool enc_put_bits(uint64_t& x, Emit& emit, uint32_t val) {
    const uint64_t x_max = (kRansL >> kBypassPrecision) << 32;
    if (x >= x_max) {
        if (!emit(uint32_t(x))) return false;
        x >>= 32;
    }
    x = (x << kBypassPrecision) | val;
    return true;
}

// One (symbol, CDF row) element, pushed in reverse: escape digits high first, the digit count's remainder, its 15s, and
// last the CDF symbol.  cdf: the row's `size` entries (size <= stride is the caller's check).
RANS_HD_TEMPLATE
template <class Emit>
RANS_HD int encode_element_reversed(uint64_t& x, Emit& emit, int32_t symbol, const int32_t* cdf, int32_t size, int32_t offset) {
    const int32_t max_value = size - 2;
    if (max_value < 0) return kInvalid;
    int32_t value = symbol - offset;
    uint32_t raw = 0;
    bool escape = false;
    if (value < 0) {
        raw = uint32_t(-2 * int64_t(value) - 1);
        value = max_value;
        escape = true;
    } else if (value >= max_value) {
        raw = uint32_t(2 * (int64_t(value) - max_value));
        value = max_value;
        escape = true;
    }
    const int32_t lo = cdf[value], hi = cdf[value + 1];
    if (hi <= lo) return kInvalid;                              // zero-probability symbol: the table is broken
    if (escape) {
        int32_t ndig = 0;
        while (ndig < kMaxDigits && (raw >> (ndig * kBypassPrecision)) != 0) ++ndig;
        for (int32_t j = ndig; j-- > 0;)
            if (!enc_put_bits(x, emit, (raw >> (j * kBypassPrecision)) & kMaxBypass)) return kFull;
        if (!enc_put_bits(x, emit, uint32_t(ndig % kMaxBypass))) return kFull;
        for (int32_t q = ndig / kMaxBypass; q > 0; --q)
            if (!enc_put_bits(x, emit, kMaxBypass)) return kFull;
    }
    return enc_put(x, emit, uint32_t(lo), uint32_t(hi - lo)) ? kOk : kFull;
}

// Reads one stream of 32-bit words forward.  `ok` drops when a renormalisation needs a word past `end`.
struct Decoder {
    const uint32_t* w;
    int64_t p, end;
    uint64_t x;
    bool ok;

    // the first two words are the encoder's final state (low half, high half)
    RANS_HD void init(const uint32_t* words, int64_t begin, int64_t stop) {
        w = words; p = begin; end = stop; ok = stop - begin >= 2;
        x = 0;
        if (ok) {
            x = uint64_t(w[p]) | (uint64_t(w[p + 1]) << 32);
            p += 2;
        }
    }
    RANS_HD void renorm() {
        if (x < kRansL) {
            if (p < end) x = (x << 32) | w[p++];
            else ok = false;
        }
    }
    RANS_HD uint32_t get_bits(uint32_t nbits) {
        const uint32_t v = uint32_t(x & ((uint64_t(1) << nbits) - 1));
        x >>= nbits;
        renorm();
        return v;
    }
};

// Decodes one element with CDF row `cdf` (size entries).  Returns false on a truncated or corrupt stream.
RANS_HD bool decode_element(Decoder& d, const int32_t* cdf, int32_t size, int32_t offset, int32_t& out) {
    const int32_t max_value = size - 2;
    const uint32_t cum = uint32_t(d.x & ((uint64_t(1) << kPrecision) - 1));
    // last entry <= cum (entries are increasing; the table is short: binary search)
    int lo = 0, hi = size - 1;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (uint32_t(cdf[mid]) <= cum) lo = mid;
        else hi = mid;
    }
    const uint32_t start = uint32_t(cdf[lo]), freq = uint32_t(cdf[lo + 1] - cdf[lo]);
    d.x = freq * (d.x >> kPrecision) + (d.x & ((uint64_t(1) << kPrecision) - 1)) - start;
    d.renorm();
    int32_t value = lo;
    if (value == max_value) {
        int32_t v = int32_t(d.get_bits(kBypassPrecision));
        int32_t ndig = v;
        while (v == kMaxBypass && d.ok) {
            v = int32_t(d.get_bits(kBypassPrecision));
            ndig += v;
        }
        if (ndig > kMaxDigits) return false;                    // no encoder writes more digits than a uint32 has
        uint32_t raw = 0;
        for (int32_t j = 0; j < ndig; ++j) raw |= d.get_bits(kBypassPrecision) << (j * kBypassPrecision);
        value = int32_t(raw >> 1);
        if (raw & 1) value = -value - 1;
        else value += max_value;
    }
    out = value + offset;
    return d.ok;
}

}  // namespace rans
}  // namespace b200
