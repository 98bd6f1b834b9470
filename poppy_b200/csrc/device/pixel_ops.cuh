// Per-pixel arithmetic shared by the tiled kernels: 8-bit <-> float conversions as cv::Mat::convertTo evaluates
// them, and the per-frame blend mask. Every helper is exact with respect to the reference's CPU arithmetic
// (SURVEY.md Appendix A.7); the tricks below only change which GPU pipe does the work.
#pragma once

#include "common.cuh"

namespace poppy {

constexpr float kInv255 = (float)(1.0 / 255.0);

// convertTo(CV_32F, 1/255) of byte `c` of a packed word: float(v) * float(1/255.0), rounded once
// (OCV core/src/convert_scale.simd.hpp:91-125). Instead of an integer->float conversion (quarter-rate pipe) the byte
// is dropped into the mantissa of 2^23 (one PRMT: 0x4B0000vv = 2^23 + v exactly) and a single FMA computes
// (2^23 + v) * k - 2^23 * k = v * k with one rounding; 2^23 * k is exact, so the result equals __fmul_rn((float)v, k).
__device__ __forceinline__ float unit_from_byte(uint32_t word, int c) {
    const float m = __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7440u | (uint32_t)c));
    return fmaf(m, kInv255, -8388608.0f * kInv255);
}

// m2 = 1 - gray(gabor2) of one pixel, the mask basis (reference src/algo.cpp:250-252). RGB2Gray<float>
// (OCV imgproc/src/color_rgb.simd.hpp:594-642) runs per row: the 8-lane vector body evaluates fma(r,cr, fma(g,cg, b*cb));
// the scalar tail (last w%8 pixels) is contracted to fma(r,cr, fma(b,cb, g*cg)). body: x < (w & ~7).
__device__ __forceinline__ float mask_basis_px(float b, float g, float r, bool body) {
    const float gray = body ? fmaf(r, 0.299f, fmaf(g, 0.587f, __fmul_rn(b, 0.114f)))
                            : fmaf(r, 0.299f, fmaf(b, 0.114f, __fmul_rn(g, 0.587f)));
    return __fsub_rn(1.0f, gray);
}

// lbmask of one pixel (reference src/algo.cpp:255-258): addWeighted(ones, 1-mr, m2, -mr) evaluates
// alpha + round(m2 * beta) in double and narrows (OCV core/src/arithm.simd.hpp:1161-1204,1721-1730), then the two
// setTo() clamps.
__device__ __forceinline__ float blend_mask(float m2, double alpha, double beta) {
    const float m = __double2float_rn(__dadd_rn(alpha, __dmul_rn((double)m2, beta)));
    return m < 0.f ? 0.f : (m > 1.f ? 1.f : m);
}

// convertTo(CV_8U, 255) of one value: saturate_cast<uchar>(cvRound(v * 255.f)) (convert_scale.simd.hpp:233,
// saturate.hpp:105). Clamping to [0, 255] before rounding is equivalent (rounding is monotonic and fixes 0 and 255;
// NaN -> 0 on both routes), and adding 1.5 * 2^23 rounds half-to-even at integer granularity, leaving the byte in the
// low mantissa bits - no float->int conversion (quarter-rate pipe) is issued. Returns the float whose low byte is
// the result; pack with pack_u8x4().
__device__ __forceinline__ float u8_magic(float v) {
    float t = __fmul_rn(v, 255.f);
    t = fminf(fmaxf(t, 0.f), 255.f);
    return __fadd_rn(t, 12582912.0f);
}
__device__ __forceinline__ uint32_t pack_u8x4(float a, float b, float c, float d) {
    const uint32_t lo = __byte_perm(__float_as_uint(a), __float_as_uint(b), 0x0040);
    const uint32_t hi = __byte_perm(__float_as_uint(c), __float_as_uint(d), 0x0040);
    return __byte_perm(lo, hi, 0x5410);
}

}  // namespace poppy
