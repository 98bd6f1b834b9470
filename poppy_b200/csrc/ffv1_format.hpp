// The one FFV1 configuration this project writes (host and device code share it; DESIGN §9.1):
// version 3 (micro 4), range coder with the default state-transition table, RGB via JPEG2000-RCT, 8 bits, no alpha, no slice
// CRCs, intra only, one quant-table set (libavcodec's quant11 with context model 0) for both context planes, initial states 128.
#pragma once
#include <stdint.h>

namespace poppy {
namespace ffv1 {

constexpr int kContexts = (11 * 11 * 11 + 1) / 2;     // 666: q(L-LT) + 11 q(LT-T) + 121 q(T-RT), folded by sign
constexpr int kStateBytes = 32;                        // range-coder states of one context
constexpr int kMaxSlicesH = 32, kMaxSlicesV = 32;      // 1024 slices: the most libavcodec's decoder accepts
// Worst case of one sample, in bytes (DESIGN §9.1): a 9-bit folded residual takes at most 19 binary decisions (zero flag, 8 + 1
// exponent decisions, 8 mantissa bits, sign). Every state stays in [8, 248], so a decision keeps at least floor(r * 8 / 256) of
// a range r >= 256, i.e. costs at most log2(8192 / 225) < 5.19 bits; 19 of them are < 98.7 bits < 12.34 bytes.
constexpr int kWorstBytesPer3Samples = 38;             // > 3 * 12.34 bytes: one pixel
constexpr int kSliceAllowance = 64;                    // keyframe bit, slice header, termination and the 24-bit slice size

// Slices of about 128 x 96 pixels (8-16 k), at most 32 x 32, never more columns than w or rows than h.
inline void slice_grid(int w, int h, int* nh, int* nv) {
    int a = (w + 64) / 128, b = (h + 48) / 96;
    a = a < 1 ? 1 : a; b = b < 1 ? 1 : b;
    a = a > kMaxSlicesH ? kMaxSlicesH : a; b = b > kMaxSlicesV ? kMaxSlicesV : b;
    *nh = a > w ? w : a; *nv = b > h ? h : b;
}

// libavcodec's ff_build_rac_states(c, 0.05 * 2^32, 256 - 8): the default state-transition table.
inline void build_states(uint8_t zero[256], uint8_t one[256]) {
    const int64_t kOne = 1LL << 32, factor = (int64_t)(0.05 * (double)(1LL << 32));
    const int max_p = 256 - 8;
    int ones[256] = {0};
    int64_t p = kOne / 2;
    int last = 0;
    for (int i = 0; i < 128; ++i) {
        int p8 = (int)((256 * p + kOne / 2) >> 32);
        if (p8 <= last) p8 = last + 1;
        if (last && last < 256 && p8 <= max_p) ones[last] = p8;
        p += ((kOne - p) * factor + kOne / 2) >> 32;
        last = p8;
    }
    for (int i = 256 - max_p; i <= max_p; ++i) {
        if (ones[i]) continue;
        p = ((int64_t)i * kOne + 128) >> 8;
        p += ((kOne - p) * factor + kOne / 2) >> 32;
        int p8 = (int)((256 * p + kOne / 2) >> 32);
        if (p8 <= i) p8 = i + 1;
        if (p8 > max_p) p8 = max_p;
        ones[i] = p8;
    }
    for (int i = 0; i < 256; ++i) { one[i] = (uint8_t)ones[i]; zero[i] = 0; }
    for (int i = 1; i < 255; ++i) zero[i] = (uint8_t)(256 - ones[256 - i]);
}

// quant11 of libavcodec (ffv1enc.c) for a difference d (mod 256): runs of 1, 1, 3, 7, 23 and 93 indices take 0..5, mirrored
// with a minus sign for negative d (-128 -> -5).
#if defined(__CUDACC__)
__host__ __device__
#endif
inline int quant11(int d) {
    const int s = (int8_t)(uint8_t)d;
    const int a = s < 0 ? -s : s;
    const int q = a == 0 ? 0 : a == 1 ? 1 : a < 5 ? 2 : a < 12 ? 3 : a < 35 ? 4 : 5;
    return s < 0 ? -q : q;
}

}  // namespace ffv1
}  // namespace poppy
