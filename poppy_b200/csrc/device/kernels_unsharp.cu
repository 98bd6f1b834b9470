// Kernel group 4 — unsharp_mask(lapBlend, 1, amount, 0.3) fused with the final convertTo(CV_8U, 255).
// reference src/util.cpp:113-148, src/algo.cpp:263-265
//
//   GaussianBlur(sigma 1) -> 9 taps, separable, BORDER_REFLECT_101. Row filter and symmetric column filter both
//   run as FMA chains in OpenCV's FMA-dispatched translation unit:
//     row:    s = k[-4]*x[-4]; s = fma(x[j], k[j], s), j = -3..4       (OCV imgproc/src/filter.simd.hpp:1663-1681,2477-2487)
//     column: s = fma(k0, t0, 0); s = fma(k[j], t[+j] + t[-j], s), j = 1..4   (filter.simd.hpp:1909-1960)
//   except for the last (3*w) % 8 interleaved elements of every row, which fall to the generic scalar loops
//   (filter.simd.hpp:2477-2487, 2753-2759); the reference build does not contract those: products and sums are
//   rounded separately there.
//   diff = x - blur; 3x3 per-channel median with replicated border (median_blur.simd.hpp:677-745);
//   where ||diff||_2 >= 0.3 (cv::norm of a Vec3f: double accumulation + sqrt): x + amount*diff, else x
//   (src/util.cpp:135-145, unfused); then cvRound(v*255) saturated to 8 bits (convert_scale.simd.hpp, saturate.hpp:105).
//
// Design: one CTA walks a 120-column strip of the frame downwards, 8 rows per step, keeping three 16-row rings in
// shared memory (the input rows, their row-pass results, and the blur differences), so the 9x9 + 3x3 footprint costs
// no vertical halo and every input value is read from global memory once (plus 8/120 horizontally). The step loop is
// unrolled by two: rows advance by 8 per step, so with 16-row rings every ring slot is a compile-time constant of the
// step parity and shared-memory accesses need no address arithmetic. Per step:
//   R  one warp per (row, channel): load 4 px per lane, exchange the horizontal neighbours through the input ring,
//      row pass -> row-pass ring
//   C  column pass with a 12-row register window per thread (4 columns x 4 rows), diff -> diff ring; a bit mask per
//      (row, channel) records which 4-px groups hold any |diff| >= 0.17
//   M  8 rows x 30 groups: where no flagged group touches the 3x3 window the median cannot reach the 0.3 threshold
//      (|median| <= max |diff| < 0.3/sqrt(3)), so the pixel is the input; otherwise the exact median/norm/sharpen runs.
//      Rounding to 8 bits uses the magic-number trick of pixel_ops.cuh; rows are written as three 32-bit words per lane.

#include "common.cuh"
#include "kernels.cuh"
#include "pixel_ops.cuh"

namespace poppy {

namespace {

constexpr int US_W = 120;            // output columns per strip
constexpr int US_CW = 128;           // computed columns x0-4 .. x0+123
constexpr int US_XW = 136;           // staged input columns x0-8 .. x0+127
constexpr int US_STEP = 8;           // rows per step
constexpr int US_PF_ROWS = US_STEP;  // L2 prefetch distance of the row stage (one step; two bring nothing more)
constexpr int US_RING = 16;          // ring depth (rows) of the three shared-memory rings
constexpr int US_CHUNK = 216;        // default rows per CTA (a launch parameter: the sparse pass over flagged chunks uses fewer)
constexpr size_t US_SMEM = ((size_t)US_RING * 3 * US_XW + 2 * (size_t)US_RING * 3 * US_CW) * sizeof(float) +
                           US_RING * 4 * sizeof(uint32_t);
constexpr float US_FLAG_T = 0.17f;   // 3 * 0.17^2 = 0.0867 < 0.09: below this no median can reach the threshold

// getGaussianKernel(9, 1, CV_32F) (bit-exact kernel, OCV imgproc/src/smooth.dispatch.cpp:81-198): centre .. edge
__device__ __forceinline__ float gk(int j) {
    j = j < 0 ? -j : j;
    const unsigned bits = j == 0 ? 0x3ecc4252u : j == 1 ? 0x3e77c75du : j == 2 ? 0x3d5d25cdu : j == 3 ? 0x3b913926u : 0x390c54e2u;
    return __uint_as_float(bits);
}

#define POPPY_SORT2(a, b) { float lo_ = fminf(a, b); b = fmaxf(a, b); a = lo_; }
__device__ __forceinline__ float median9(float p0, float p1, float p2, float p3, float p4, float p5, float p6, float p7,
                                         float p8) {
    POPPY_SORT2(p1, p2) POPPY_SORT2(p4, p5) POPPY_SORT2(p7, p8) POPPY_SORT2(p0, p1) POPPY_SORT2(p3, p4)
    POPPY_SORT2(p6, p7) POPPY_SORT2(p1, p2) POPPY_SORT2(p4, p5) POPPY_SORT2(p7, p8) POPPY_SORT2(p0, p3)
    POPPY_SORT2(p5, p8) POPPY_SORT2(p4, p7) POPPY_SORT2(p3, p6) POPPY_SORT2(p1, p4) POPPY_SORT2(p2, p5)
    POPPY_SORT2(p4, p7) POPPY_SORT2(p4, p2) POPPY_SORT2(p6, p4) POPPY_SORT2(p4, p2)
    return p4;
}
#undef POPPY_SORT2

// row filter at one pixel, fused (vector body) or unfused (scalar tail) — taps t[0..8] left to right
__device__ __forceinline__ float row9(const float* t, bool fused) {
    float s = __fmul_rn(gk(-4), t[0]);
    if (fused) {
#pragma unroll
        for (int j = 1; j < 9; ++j) s = fmaf(t[j], gk(j - 4), s);
    } else {
#pragma unroll
        for (int j = 1; j < 9; ++j) s = __fadd_rn(s, __fmul_rn(gk(j - 4), t[j]));
    }
    return s;
}

// the fused symmetric column filter on two adjacent columns at once (sm_100 FADD2 / FFMA2: both halves individually rounded,
// so the results are those of col9(..., true) per column)
__device__ __forceinline__ float2 col9_fused2(float2 w0, float2 w1, float2 w2, float2 w3, float2 w4, float2 w5, float2 w6, float2 w7,
                                              float2 w8) {
    float2 s = __ffma2_rn(make_float2(gk(0), gk(0)), w4, make_float2(0.f, 0.f));
    s = __ffma2_rn(make_float2(gk(1), gk(1)), __fadd2_rn(w5, w3), s);
    s = __ffma2_rn(make_float2(gk(2), gk(2)), __fadd2_rn(w6, w2), s);
    s = __ffma2_rn(make_float2(gk(3), gk(3)), __fadd2_rn(w7, w1), s);
    return __ffma2_rn(make_float2(gk(4), gk(4)), __fadd2_rn(w8, w0), s);
}

// symmetric column filter — w[0..8] top to bottom
__device__ __forceinline__ float col9(float w0, float w1, float w2, float w3, float w4, float w5, float w6, float w7,
                                      float w8, bool fused) {
    if (fused) {
        float s = fmaf(gk(0), w4, 0.f);
        s = fmaf(gk(1), __fadd_rn(w5, w3), s);
        s = fmaf(gk(2), __fadd_rn(w6, w2), s);
        s = fmaf(gk(3), __fadd_rn(w7, w1), s);
        return fmaf(gk(4), __fadd_rn(w8, w0), s);
    }
    float s = __fadd_rn(__fmul_rn(gk(0), w4), 0.f);
    s = __fadd_rn(s, __fmul_rn(gk(1), __fadd_rn(w5, w3)));
    s = __fadd_rn(s, __fmul_rn(gk(2), __fadd_rn(w6, w2)));
    s = __fadd_rn(s, __fmul_rn(gk(3), __fadd_rn(w7, w1)));
    return __fadd_rn(s, __fmul_rn(gk(4), __fadd_rn(w8, w0)));
}

__device__ __forceinline__ void us_cp_async16(float* smem_dst, const float* gmem_src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src) : "memory");
}

// Per-thread constants of the strip kernel.
struct UsThread {
    int w, h, lane, warp, gx0, x0, Y0, Y1, tail_from;
    bool in_img;          // the lane's 4 computed columns start inside the image
    bool lane_fast;       // all 12 row-pass taps inside the image and in the vector-body region
    bool halo;            // lane 0 / 1 stage the 4 columns left / right of the computed range
    int halo_goff;        // their offset from column gx0 in global memory ...
    int halo_soff;        // ... and their float offset in an input-ring row
    int rfl_dst, rfl_src; // border strips: staged slot outside the image this lane fills, and the staged slot it mirrors (-1: none)
};

constexpr int US_XROW = 3 * US_XW, US_CROW = 3 * US_CW;      // floats per ring row (3 channels)

// R: row pass of virtual row vb + 5 + warp, all three channels; the ring slot is passed in. INTERIOR (a CTA-uniform
// property of the strip): every lane's taps lie inside the image and in the vector-body region, so no border logic.
// All global loads of the row (3 channels, plus the halo groups of lanes 0/1) are issued before the first one is
// consumed, so a warp exposes one memory latency per row instead of three. In border strips the staged columns that lie
// outside the image are then filled by reflection from the staged row itself (BORDER_REFLECT_101), after which border
// lanes run the same row filter as interior ones.
template <bool INTERIOR>
__device__ __forceinline__ void us_row_pass(const UsThread& T, const float* __restrict__ img, int pitch, size_t stride,
                                            float* xs_row, float* rp_row, int v) {
    const float* __restrict__ row = img + (size_t)reflect101(v, T.h) * pitch + T.gx0;
    if (INTERIOR) {
        // the row this warp stages in the NEXT step (8 rows down): start it on its way from HBM to L2 now, so that the
        // loads below - whose latency nothing in this warp can cover - find it there (shared memory leaves no L1 to
        // prefetch into)
        const float* __restrict__ nxt = img + (size_t)reflect101(v + US_PF_ROWS, T.h) * pitch + T.gx0;
#pragma unroll
        for (int c = 0; c < 3; ++c) asm volatile("prefetch.global.L2 [%0];" ::"l"(nxt + c * stride));
    }
    float4 own[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        own[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (INTERIOR || T.in_img) own[c] = __ldg(reinterpret_cast<const float4*>(row + c * stride));
        // the halo groups go straight to shared memory (LDGSTS): no registers held across the latency
        if (T.halo) us_cp_async16(xs_row + c * US_XW + T.halo_soff, row + c * stride + T.halo_goff);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c)
        if (INTERIOR || T.in_img) *reinterpret_cast<float4*>(xs_row + c * US_XW + 4 + 4 * T.lane) = own[c];
    asm volatile("cp.async.wait_all;\n" ::: "memory");
    __syncwarp();
    if (!INTERIOR && T.rfl_dst >= 0) {
#pragma unroll
        for (int c = 0; c < 3; ++c) xs_row[c * US_XW + T.rfl_dst] = xs_row[c * US_XW + T.rfl_src];
    }
    if (!INTERIOR) __syncwarp();
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float* xrow = xs_row + c * US_XW;
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        if (INTERIOR || T.lane_fast) {
            const float4 lft = *reinterpret_cast<const float4*>(xrow + 4 * T.lane);
            const float4 rgt = *reinterpret_cast<const float4*>(xrow + 8 + 4 * T.lane);
            const float t[12] = {lft.x, lft.y, lft.z, lft.w, own[c].x, own[c].y, own[c].z, own[c].w, rgt.x, rgt.y, rgt.z, rgt.w};
            o.x = row9(t + 0, true); o.y = row9(t + 1, true); o.z = row9(t + 2, true); o.w = row9(t + 3, true);
        } else if (T.in_img) {
            // partial groups at the right image edge and the scalar-tail elements: per pixel, taps from the staged row
            float r[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
            for (int i = 0; i < 4; ++i) {
                const int gx = T.gx0 + i;
                if (gx >= T.w) continue;
                if (T.w == 1) { r[i] = xrow[4 + 4 * T.lane + i]; continue; }      // GaussianBlur shrinks the kernel to [1] on a 1-pixel axis
                float t[9];
#pragma unroll
                for (int j = 0; j < 9; ++j) t[j] = xrow[4 * T.lane + i + j];
                r[i] = row9(t, 3 * gx + c < T.tail_from);
            }
            o = make_float4(r[0], r[1], r[2], r[3]);
        }
        *reinterpret_cast<float4*>(rp_row + c * US_CW + 4 * T.lane) = o;
    }
}

// C: column pass + diff of rows vb+1+4*HF .. +3 for channel c; every ring slot is a compile-time constant.
template <bool INTERIOR, int PAR, int HF>
__device__ __forceinline__ void us_col_pass(const UsThread& T, const float* rp_t, const float* xs_t, float* df_t,
                                            uint32_t* fl_c, int vb, int c) {
    constexpr int K0 = 8 * PAR + 4 * HF - 3;                 // window row j lives in ring slot (K0 + j) & 15
    const int v0 = vb + 1 + 4 * HF;
    const int lo = max(T.Y0 - 1, 0), hi = min(T.Y1, T.h - 1);          // diff rows this CTA needs: [lo, hi]
    if (v0 + 3 < lo || v0 > hi) return;
    float4 win[12];
#pragma unroll
    for (int j = 0; j < 12; ++j) win[j] = *reinterpret_cast<const float4*>(rp_t + ((K0 + j) & 15) * US_CROW);
    const bool fused = INTERIOR || 3 * (T.gx0 + 3) + c < T.tail_from;         // whole group in the vector body
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int slot = (K0 + 4 + i) & 15;
        const int v = v0 + i;
        if (v < lo || v > hi) continue;                            // warp-uniform
        float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
        bool big = false;
        if (INTERIOR || T.in_img) {
            float4 b;
            if (!INTERIOR && T.h == 1) {
                b = win[4 + i];
            } else if (fused) {
#define POPPY_LO(k) make_float2(win[i + (k)].x, win[i + (k)].y)
#define POPPY_HI(k) make_float2(win[i + (k)].z, win[i + (k)].w)
                const float2 lo = col9_fused2(POPPY_LO(0), POPPY_LO(1), POPPY_LO(2), POPPY_LO(3), POPPY_LO(4), POPPY_LO(5), POPPY_LO(6), POPPY_LO(7), POPPY_LO(8));
                const float2 hi = col9_fused2(POPPY_HI(0), POPPY_HI(1), POPPY_HI(2), POPPY_HI(3), POPPY_HI(4), POPPY_HI(5), POPPY_HI(6), POPPY_HI(7), POPPY_HI(8));
#undef POPPY_LO
#undef POPPY_HI
                b = make_float4(lo.x, lo.y, hi.x, hi.y);
            } else {
                b.x = col9(win[i].x, win[i + 1].x, win[i + 2].x, win[i + 3].x, win[i + 4].x, win[i + 5].x, win[i + 6].x, win[i + 7].x, win[i + 8].x, 3 * (T.gx0 + 0) + c < T.tail_from);
                b.y = col9(win[i].y, win[i + 1].y, win[i + 2].y, win[i + 3].y, win[i + 4].y, win[i + 5].y, win[i + 6].y, win[i + 7].y, win[i + 8].y, 3 * (T.gx0 + 1) + c < T.tail_from);
                b.z = col9(win[i].z, win[i + 1].z, win[i + 2].z, win[i + 3].z, win[i + 4].z, win[i + 5].z, win[i + 6].z, win[i + 7].z, win[i + 8].z, 3 * (T.gx0 + 2) + c < T.tail_from);
                b.w = col9(win[i].w, win[i + 1].w, win[i + 2].w, win[i + 3].w, win[i + 4].w, win[i + 5].w, win[i + 6].w, win[i + 7].w, win[i + 8].w, 3 * (T.gx0 + 3) + c < T.tail_from);
            }
            const float4 x = *reinterpret_cast<const float4*>(xs_t + slot * US_XROW);
            {   // x - b, two columns per instruction: fma(b, -1, x) rounds the exact difference once
                const float2 dlo = __ffma2_rn(make_float2(b.x, b.y), make_float2(-1.f, -1.f), make_float2(x.x, x.y));
                const float2 dhi = __ffma2_rn(make_float2(b.z, b.w), make_float2(-1.f, -1.f), make_float2(x.z, x.w));
                d = make_float4(dlo.x, dlo.y, dhi.x, dhi.y);
            }
            // columns past the image hold padding: keep them out of the flags
            const float m0 = fabsf(d.x), m1 = (INTERIOR || T.gx0 + 1 < T.w) ? fabsf(d.y) : 0.f,
                        m2 = (INTERIOR || T.gx0 + 2 < T.w) ? fabsf(d.z) : 0.f, m3 = (INTERIOR || T.gx0 + 3 < T.w) ? fabsf(d.w) : 0.f;
            big = !(fmaxf(fmaxf(m0, m1), fmaxf(m2, m3)) < US_FLAG_T);
        }
        *reinterpret_cast<float4*>(df_t + slot * US_CROW) = d;
        const uint32_t bits = __ballot_sync(0xffffffffu, big);
        if (T.lane == 0) fl_c[slot * 4] = bits;
    }
}

// M: median / threshold / sharpen / 8-bit store of row vb + warp.
template <bool INTERIOR, int PAR>
__device__ __forceinline__ void us_emit(const UsThread& T, const float* xs, const float* df, const uint32_t* fl, int vb,
                                        float amount, double norm_thr2, uint8_t* __restrict__ dst, bool dst_words) {
    const int y = vb + T.warp, gx = T.x0 + 4 * T.lane;
    if (y >= T.Y1 || T.lane >= US_W / 4 || (!INTERIOR && gx >= T.w)) return;
    const int ym = max(y - 1, 0), yp = min(y + 1, T.h - 1);
    const int sc = (8 * PAR + T.warp) & 15, sm = (sc + (ym - y)) & 15, sp = (sc + (yp - y)) & 15;
    // computed-column group of gx is lane+1; its 3x3 windows reach groups lane .. lane+2
    const uint4 fa = *reinterpret_cast<const uint4*>(fl + sm * 4), fb = *reinterpret_cast<const uint4*>(fl + sc * 4),
                fc = *reinterpret_cast<const uint4*>(fl + sp * 4);
    const uint32_t flagged = (fa.x | fa.y | fa.z | fb.x | fb.y | fb.z | fc.x | fc.y | fc.z) & (7u << T.lane);
    const float* xrow = xs + sc * US_XROW + 8 + 4 * T.lane;
    float4 px[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) px[c] = *reinterpret_cast<const float4*>(xrow + c * US_XW);
    float v[3][4] = {{px[0].x, px[0].y, px[0].z, px[0].w}, {px[1].x, px[1].y, px[1].z, px[1].w}, {px[2].x, px[2].y, px[2].z, px[2].w}};
    const int npx = INTERIOR ? 4 : min(4, T.w - gx);
    if (flagged) {
#pragma unroll 1
        for (int i = 0; i < npx; ++i) {
            const int cc = 4 + 4 * T.lane + i;                            // column in the diff ring
            const int cm = max(gx + i - 1, 0) - (T.x0 - 4), cp = min(gx + i + 1, T.w - 1) - (T.x0 - 4);
            float med[3];
            double nn = 0.0;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float* d0 = df + sm * US_CROW + c * US_CW;
                const float* d1 = df + sc * US_CROW + c * US_CW;
                const float* d2 = df + sp * US_CROW + c * US_CW;
                med[c] = median9(d0[cm], d0[cc], d0[cp], d1[cm], d1[cc], d1[cp], d2[cm], d2[cc], d2[cp]);
                nn = __dadd_rn(nn, __dmul_rn((double)med[c], (double)med[c]));
            }
            if (nn >= norm_thr2) {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float add = __fmul_rn(amount, med[c]);
                    // static indexing keeps v[][] in registers
                    if (i == 0) v[c][0] = __fadd_rn(v[c][0], add);
                    else if (i == 1) v[c][1] = __fadd_rn(v[c][1], add);
                    else if (i == 2) v[c][2] = __fadd_rn(v[c][2], add);
                    else v[c][3] = __fadd_rn(v[c][3], add);
                }
            }
        }
    }
    float q[3][4];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < 4; ++i) q[c][i] = u8_magic(v[c][i]);
    uint8_t* drow = dst + ((size_t)y * T.w + gx) * 3;
    if (INTERIOR || (dst_words && npx == 4)) {
        uint32_t* d32 = reinterpret_cast<uint32_t*>(drow);
        d32[0] = pack_u8x4(q[0][0], q[1][0], q[2][0], q[0][1]);
        d32[1] = pack_u8x4(q[1][1], q[2][1], q[0][2], q[1][2]);
        d32[2] = pack_u8x4(q[2][2], q[0][3], q[1][3], q[2][3]);
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (i < npx) {
#pragma unroll
                for (int c = 0; c < 3; ++c) drow[3 * i + c] = (uint8_t)(__float_as_uint(q[c][i]) & 255u);
            }
    }
}

// One step (8 rows) of the strip walk; PAR = step parity, which fixes every ring slot at compile time
// (rows advance by 8 per step, the rings hold 16 rows).
template <bool INTERIOR, int PAR>
__device__ __forceinline__ void us_step(const UsThread& T, int s, const float* __restrict__ img, int pitch, size_t stride,
                                        float* xs, float* rp, float* df, uint32_t* fl, float amount, double norm_thr2,
                                        uint8_t* __restrict__ dst, bool dst_words) {
    const int vb = T.Y0 + US_STEP * s;
    {   // R: virtual row vb + 5 + warp
        const int v = vb + 5 + T.warp;
        if (v >= T.Y0 - 5 && v <= T.Y1 + 4) {
            const int slot = (8 * PAR + 5 + T.warp) & 15;
            us_row_pass<INTERIOR>(T, img, pitch, stride, xs + slot * US_XROW, rp + slot * US_CROW, v);
        }
    }
    __syncthreads();
    if (T.warp < 6) {
        const int c = T.warp >> 1;
        const float* rp_t = rp + c * US_CW + 4 * T.lane;
        const float* xs_t = xs + c * US_XW + 4 + 4 * T.lane;
        float* df_t = df + c * US_CW + 4 * T.lane;
        if (T.warp & 1) us_col_pass<INTERIOR, PAR, 1>(T, rp_t, xs_t, df_t, fl + c, vb, c);
        else us_col_pass<INTERIOR, PAR, 0>(T, rp_t, xs_t, df_t, fl + c, vb, c);
    }
    __syncthreads();
    if (s >= 0) us_emit<INTERIOR, PAR>(T, xs, df, fl, vb, amount, norm_thr2, dst, dst_words);
    __syncthreads();
}

}  // namespace

// block 256; grid (ceil(w/120), ceil(h/216), frames); dynamic shared memory US_SMEM.
// norm_thr2: smallest double whose sqrt is >= (double)0.3f.
__global__ void __launch_bounds__(256, 3)
k_unsharp_strip(const float* __restrict__ lap, int w, int h, int pitch, size_t stride, const FrameParams* __restrict__ fp,
                double norm_thr2, uint8_t* __restrict__ frames_base, size_t frame_bytes, int chunk_rows,
                const unsigned char* __restrict__ chunk_flags) {
    extern __shared__ __align__(16) float smem_dyn[];
    float* xs = smem_dyn;                                        // [US_RING][3][US_XW]  input rows (virtual, reflected)
    float* rp = xs + US_RING * US_XROW;                          // [US_RING][3][US_CW]  row-pass results
    float* df = rp + US_RING * US_CROW;                          // [US_RING][3][US_CW]  x - blur
    uint32_t* fl = reinterpret_cast<uint32_t*>(df + US_RING * US_CROW);      // [US_RING][4] flagged 4-px groups per diff row, channel

    const int f = blockIdx.z;
    if (chunk_flags && !chunk_flags[((size_t)f * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x]) return;    // calm chunk
    UsThread T;
    T.w = w; T.h = h;
    T.x0 = blockIdx.x * US_W; T.Y0 = blockIdx.y * chunk_rows; T.Y1 = min(T.Y0 + chunk_rows, h);
    T.warp = threadIdx.x >> 5; T.lane = threadIdx.x & 31;
    T.tail_from = 3 * w - (3 * w) % 8;       // first interleaved element handled by the scalar filter loops
    T.gx0 = T.x0 - 4 + 4 * T.lane;           // this lane's 4 computed columns
    T.in_img = T.gx0 >= 0 && T.gx0 < w;
    // the lane's 4 pixels inside the image, none of them in the scalar-tail region (taps outside the image are
    // mirrored into the staged row, see us_row_pass)
    T.lane_fast = T.gx0 >= 0 && T.gx0 + 3 <= w - 1 && 3 * (T.gx0 + 3) + 2 < T.tail_from && w > 1;
    // staged slot k of a row holds column x0 - 8 + k; lanes 0-7 mirror columns -8..-1, lanes 8-15 columns w..w+7
    T.rfl_dst = T.rfl_src = -1;
    if (T.lane < 8 && T.x0 == 0 && w > 1) { T.rfl_dst = T.lane; T.rfl_src = reflect101(T.lane - 8, w) + 8; }
    if (T.lane >= 8 && T.lane < 16 && w > 1) {
        const int col = w + T.lane - 8;
        if (col <= T.x0 + 127 && col >= T.x0 - 8) { T.rfl_dst = col - T.x0 + 8; T.rfl_src = reflect101(col, w) - T.x0 + 8; }
    }
    T.halo = (T.lane == 0 && T.x0 - 8 >= 0) || (T.lane == 1 && T.x0 + 124 < w);
    T.halo_goff = T.lane == 0 ? -4 : 124;    // lane 0: columns x0-8.. (gx0 = x0-4); lane 1: columns x0+124.. (gx0 = x0)
    T.halo_soff = T.lane == 0 ? 0 : US_XW - 4;
    const float* __restrict__ img = lap + (size_t)f * 3 * stride;
    const FrameParams P = fp[f];
    uint8_t* __restrict__ dst = frames_base + (size_t)P.dst_slot * frame_bytes;
    const bool dst_words = (w & 3) == 0 && ((size_t)dst & 3) == 0;
    const int n_steps = div_up(T.Y1 - T.Y0, US_STEP);

    // strips whose 136 staged columns all lie inside the image, clear of the scalar-tail elements, with word-aligned
    // output rows, run the INTERIOR instantiation (no horizontal border logic at all)
    const bool interior = T.x0 - 8 >= 0 && T.x0 + 127 <= w - 1 && 3 * (T.x0 + 123) + 2 < T.tail_from && dst_words && h > 1;
    if (interior) {
        for (int s = -2; s < n_steps; s += 2) {
            us_step<true, 0>(T, s, img, pitch, stride, xs, rp, df, fl, P.amount, norm_thr2, dst, dst_words);
            if (s + 1 < n_steps) us_step<true, 1>(T, s + 1, img, pitch, stride, xs, rp, df, fl, P.amount, norm_thr2, dst, dst_words);
        }
    } else {
        for (int s = -2; s < n_steps; s += 2) {
            us_step<false, 0>(T, s, img, pitch, stride, xs, rp, df, fl, P.amount, norm_thr2, dst, dst_words);
            if (s + 1 < n_steps) us_step<false, 1>(T, s + 1, img, pitch, stride, xs, rp, df, fl, P.amount, norm_thr2, dst, dst_words);
        }
    }
}

// Order-dependent 64-bit checksum: per-block FNV-1a over 8-byte words folded with a position weight, atomically
// xor-added. Used for "checksum of checksums" parity at full size without copying frames to the host.
__global__ void k_checksum(const uint8_t* __restrict__ data, size_t bytes, unsigned long long* __restrict__ out) {
    unsigned long long acc = 0;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < bytes; i += stride) {
        unsigned long long v = (unsigned long long)data[i] + 1ull;
        unsigned long long k = (i + 0x9E3779B97F4A7C15ull) * 0xBF58476D1CE4E5B9ull;
        k ^= k >> 29;
        acc += v * (k | 1ull);
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

// ---- calm analysis (see EmitCtx in kernels_pyramid.cu) ----------------------------------------------------------------
// k_calm_scan bounds the unit second differences of lapBlend from the frame bytes q the fused collapse stored. Per 4x8
// block it records hx = max |floor((q[x-1] + q[x+1]) / 2) - q[x]| and hy (the same along y; neighbours reflected at the
// image border like the blur's BORDER_REFLECT_101). |q[-1] + q[+1] - 2 q[0]| <= 2 h + 1, and |255 x - q| <= 0.5 (+ 0.255
// where the block's clamp excess is tolerated), so the second differences of x are below (2 h + 3.02) / 255. A pixel is
// calm when, over the blocks within 2 block columns / 1 block row (8 pixels each way; its median + blur footprint spans 5
// columns and 4 rows of second differences), max hx + max hy <= CALM_SUM: then
//     |x - blur| <= 0.49997 ((2 hx + 3.02) + (2 hy + 3.02)) / 255 + rounding (< 1e-5) < 0.1732,
// and no 3x3 median can reach norm 0.3 (3 * 0.1732^2 < 0.09).
constexpr int CALM_SUM = 40;
static_assert(UNSHARP_STRIP_W == US_W, "strip width");
static_assert((2 * CALM_SUM + 2 * 3.02) / 255.0 * 0.49997 < 0.1731, "calm bound");

// |floor-avg(a, c) - b| of four bytes at once
__device__ __forceinline__ unsigned calm_dev4(unsigned a, unsigned b, unsigned c) {
    return __vabsdiffu4((a & c) + (((a ^ c) & 0xFEFEFEFEu) >> 1), b);
}

// block (32, 4); grid (ceil(w/128), ceil(h/64), frames). Requires w % 4 == 0, w >= 8, h >= 2 (the launcher flags everything
// otherwise). A lane owns 4 pixels = 3 words of every row and walks 16 rows (two blocks of the table) with a three-row
// window; the bytes 3 to the left / right of its own come from the neighbouring lanes' words. The running maxima are kept
// as 16-bit SIMD lanes (even bytes | odd bytes << 8: VIMNMX.U16x2).
__global__ void __launch_bounds__(128)
k_calm_scan(const uint8_t* __restrict__ frames_base, size_t frame_bytes, const FrameParams* __restrict__ fp, int w, int h,
            const unsigned char* __restrict__ ex, int ex_pitch, size_t ex_stride, int bw, int bh,
            uchar2* __restrict__ block_dev) {
    const int f = blockIdx.z, lane = threadIdx.x;
    const int x = blockIdx.x * 128 + 4 * lane, y0 = (blockIdx.y * 4 + threadIdx.y) * 16;
    if (y0 >= h) return;
    const bool active = x < w;
    const int xc = active ? x : w - 4;                        // inactive lanes shadow the last pixel group
    const uint8_t* __restrict__ frame = frames_base + (size_t)fp[f].dst_slot * frame_bytes;
    const size_t row_bytes = (size_t)w * 3;
    auto load = [&](int y, unsigned (&wd)[5]) {
        y = y < 0 ? -y : (y >= h ? 2 * h - 2 - y : y);       // BORDER_REFLECT_101
        const unsigned* __restrict__ p = reinterpret_cast<const unsigned*>(frame + (size_t)y * row_bytes + (size_t)xc * 3);
        wd[1] = __ldg(p); wd[2] = __ldg(p + 1); wd[3] = __ldg(p + 2);
        unsigned l = __shfl_up_sync(0xffffffffu, wd[3], 1), r = __shfl_down_sync(0xffffffffu, wd[1], 1);
        if (lane == 0) l = xc > 0 ? __ldg(p - 1) : __byte_perm(wd[1], wd[2], 0x5433);            // pixel -1 = pixel 1
        if (lane == 31 || xc + 4 >= w) r = xc + 4 < w ? __ldg(p + 3) : __byte_perm(wd[2], wd[3], 0x4432);   // pixel w = pixel w-2
        wd[0] = l; wd[4] = r;
    };
    unsigned up[5], mid[5], dn[5];
    load(y0 - 1, up);
    load(y0, mid);
    unsigned mx_lo = 0, mx_hi = 0, my_lo = 0, my_hi = 0;
#pragma unroll 1
    for (int k = 0; k < 16; ++k) {
        const int y = y0 + k;
        if (y >= h) break;
        load(y + 1, dn);
        unsigned vx[3], vy[3];
#pragma unroll
        for (int j = 1; j <= 3; ++j) {
            vx[j - 1] = calm_dev4(__byte_perm(mid[j - 1], mid[j], 0x4321), mid[j], __byte_perm(mid[j], mid[j + 1], 0x6543));
            vy[j - 1] = calm_dev4(up[j], mid[j], dn[j]);
        }
        mx_lo = __vimax3_u16x2(mx_lo, vx[0] & 0x00FF00FFu, vx[1] & 0x00FF00FFu);
        mx_hi = __vimax3_u16x2(mx_hi, vx[0] & 0xFF00FF00u, vx[1] & 0xFF00FF00u);
        mx_lo = __vmaxu2(mx_lo, vx[2] & 0x00FF00FFu);
        mx_hi = __vmaxu2(mx_hi, vx[2] & 0xFF00FF00u);
        my_lo = __vimax3_u16x2(my_lo, vy[0] & 0x00FF00FFu, vy[1] & 0x00FF00FFu);
        my_hi = __vimax3_u16x2(my_hi, vy[0] & 0xFF00FF00u, vy[1] & 0xFF00FF00u);
        my_lo = __vmaxu2(my_lo, vy[2] & 0x00FF00FFu);
        my_hi = __vmaxu2(my_hi, vy[2] & 0xFF00FF00u);
        if ((k & 7) == 7 || y == h - 1) {
            if (active) {
                const int by = y / CALM_BLOCK_H, bx = x / CALM_BLOCK_W;
                const unsigned char* __restrict__ e = ex + (size_t)f * 3 * ex_stride + (size_t)by * ex_pitch + bx;
                unsigned hx = max(max(mx_lo & 0xFFFFu, mx_lo >> 16), max(mx_hi & 0xFFFFu, mx_hi >> 16) >> 8);
                unsigned hy = max(max(my_lo & 0xFFFFu, my_lo >> 16), max(my_hi & 0xFFFFu, my_hi >> 16) >> 8);
                if (e[0] || e[ex_stride] || e[2 * ex_stride]) hx = hy = 255u;      // out[0] left [0, 1]: its bytes say nothing
                block_dev[((size_t)f * bh + by) * bw + bx] = make_uchar2((unsigned char)hx, (unsigned char)hy);
            }
            mx_lo = mx_hi = my_lo = my_hi = 0;
        }
#pragma unroll
        for (int j = 0; j < 5; ++j) { up[j] = mid[j]; mid[j] = dn[j]; }
    }
}

// one thread per block: flagged when max hx + max hy over the blocks within 2 columns / 1 row exceeds CALM_SUM.
// grid (ceil(bw/128), bh, frames), block 128.
__global__ void k_calm_blocks(const uchar2* __restrict__ block_dev, int bw, int bh, unsigned char* __restrict__ block_flags) {
    const int bx = blockIdx.x * blockDim.x + threadIdx.x, by = blockIdx.y, f = blockIdx.z;
    if (bx >= bw) return;
    const uchar2* __restrict__ t = block_dev + (size_t)f * bh * bw;
    int hx = 0, hy = 0;
    for (int y = max(by - 1, 0); y <= min(by + 1, bh - 1); ++y)
        for (int x = max(bx - 2, 0); x <= min(bx + 2, bw - 1); ++x) {
            const uchar2 v = t[(size_t)y * bw + x];
            hx = max(hx, (int)v.x); hy = max(hy, (int)v.y);
        }
    block_flags[((size_t)f * bh + by) * bw + bx] = hx + hy > CALM_SUM ? 1 : 0;
}

// one warp per strip chunk of k_unsharp_strip: flagged when one of its blocks is; a flagged chunk also flags the level-0
// collapse tiles (128x32) its input footprint touches. grid (ceil(chunks/8), 1, frames), block 256.
__global__ void k_calm_chunks(const unsigned char* __restrict__ block_flags, int bw, int bh, int w, int h, int chunk_rows,
                              int strips, int chunks_y, unsigned char* __restrict__ chunk_flags, int tiles_x, int tiles_y,
                              unsigned char* __restrict__ tile_flags, int* __restrict__ counts,
                              unsigned long long* __restrict__ total, int force_all) {
    const int chunk = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31, f = blockIdx.z;
    if (chunk >= strips * chunks_y) return;
    const int sx = chunk % strips, cy = chunk / strips;
    const int x0 = sx * US_W, x1 = min(x0 + US_W, w), Y0 = cy * chunk_rows, Y1 = min(Y0 + chunk_rows, h);
    const int bx0 = x0 / CALM_BLOCK_W, bx1 = (x1 - 1) / CALM_BLOCK_W, by0 = Y0 / CALM_BLOCK_H, by1 = (Y1 - 1) / CALM_BLOCK_H;
    const int nbx = bx1 - bx0 + 1, n = nbx * (by1 - by0 + 1);
    bool any = force_all != 0;
    const unsigned char* __restrict__ bf = block_flags + (size_t)f * bh * bw;
    for (int i = lane; i < n && !any; i += 32) any = bf[(size_t)(by0 + i / nbx) * bw + bx0 + i % nbx] != 0;
    any = __any_sync(0xffffffffu, any);
    if (lane == 0) {
        chunk_flags[(size_t)f * strips * chunks_y + chunk] = any ? 1 : 0;
        if (any) { atomicAdd(&counts[f], 1); atomicAdd(total, 1ull); }
    }
    if (any) {
        const int tx0 = max(x0 - 8, 0) / 128, tx1 = (min(x0 + 128, w) - 1) / 128;
        const int ty0 = max(Y0 - 5, 0) / 32, ty1 = (min(Y1 + 5, h) - 1) / 32;
        const int ntx = tx1 - tx0 + 1, nt = ntx * (ty1 - ty0 + 1);
        for (int i = lane; i < nt; i += 32)
            tile_flags[((size_t)f * tiles_y + ty0 + i / ntx) * tiles_x + tx0 + i % ntx] = 1;
    }
}

void launch_calm_analysis(cudaStream_t st, const uint8_t* frames_base, size_t frame_bytes, const FrameParams* fp,
                          const unsigned char* ex, int ex_pitch, size_t ex_stride, int w, int h, int frames, int chunk_rows,
                          unsigned char* block_dev, unsigned char* block_flags, unsigned char* chunk_flags,
                          unsigned char* tile_flags, int* counts, unsigned long long* total, int force_all) {
    const int bw = div_up(w, CALM_BLOCK_W), bh = div_up(h, CALM_BLOCK_H);
    const int strips = div_up(w, US_W), chunks_y = div_up(h, chunk_rows), tiles_x = div_up(w, 128), tiles_y = div_up(h, 32);
    // the byte scan needs word-aligned rows; odd widths and tiny frames take the exact path everywhere
    if ((w & 3) != 0 || w < 8 || h < 2 || (reinterpret_cast<size_t>(frames_base) & 3) != 0 || (frame_bytes & 3) != 0) force_all = 1;
    cudaMemsetAsync(tile_flags, 0, (size_t)frames * tiles_x * tiles_y, st);
    cudaMemsetAsync(counts, 0, (size_t)frames * sizeof(int), st);
    if (!force_all) {
        k_calm_scan<<<dim3(div_up(w, 128), div_up(h, 64), frames), dim3(32, 4), 0, st>>>(
            frames_base, frame_bytes, fp, w, h, ex, ex_pitch, ex_stride, bw, bh, reinterpret_cast<uchar2*>(block_dev));
        k_calm_blocks<<<dim3(div_up(bw, 128), bh, frames), 128, 0, st>>>(reinterpret_cast<const uchar2*>(block_dev), bw, bh, block_flags);
    }
    k_calm_chunks<<<dim3(div_up(strips * chunks_y, 8), 1, frames), 256, 0, st>>>(block_flags, bw, bh, w, h, chunk_rows, strips, chunks_y,
                                                                                 chunk_flags, tiles_x, tiles_y, tile_flags, counts,
                                                                                 total, force_all);
}

void launch_unsharp_store(cudaStream_t st, const float* lap_blend, LevelDesc l, const FrameParams* fp,
                          uint8_t* frames_base, size_t frame_bytes, int frames, int chunk_rows,
                          const unsigned char* chunk_flags) {
    // smallest double s with sqrt(s) >= (double)0.3f: lets the kernel compare the squared norm (exactly
    // equivalent to "cv::norm(diff) >= threshold" with a correctly rounded sqrt)
    static const double thr2 = [] {
        const double t = (double)0.3f;
        double s = t * t;
        while (__builtin_sqrt(s) >= t) s = __builtin_nextafter(s, 0.0);
        while (__builtin_sqrt(s) < t) s = __builtin_nextafter(s, 1.0);
        return s;
    }();
    static SmemAttrOnce done;
    ensure_smem_attr(k_unsharp_strip, US_SMEM, done);
    if (chunk_rows <= 0) chunk_rows = US_CHUNK;
    k_unsharp_strip<<<dim3(div_up(l.w, US_W), div_up(l.h, chunk_rows), frames), 256, US_SMEM, st>>>(
        lap_blend, l.w, l.h, l.pitch, l.plane_stride, fp, thr2, frames_base, frame_bytes, chunk_rows, chunk_flags);
}

void launch_checksum(cudaStream_t st, const uint8_t* data, size_t bytes, unsigned long long* out) {
    int blocks = (int)((bytes + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (blocks < 1) blocks = 1;
    k_checksum<<<blocks, 256, 0, st>>>(data, bytes, out);
}

}  // namespace poppy
