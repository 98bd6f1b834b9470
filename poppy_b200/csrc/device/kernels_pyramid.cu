// Kernel group 3 — Laplacian-pyramid blend (reference src/blend.hpp:11-91) on planar float32 levels.
//
// Per frame and level k >= 1 the Gaussian pyramids are stored as 7 planes (left B,G,R, right B,G,R, mask); level 0
// is never materialised in float for the images: it is the warped 8-bit pair converted on the fly
// (src/algo.cpp:247-248). The level-0 blend mask (src/algo.cpp:250-258) is evaluated once, by the mask role of the
// level 0 -> 1 kernel, and kept as a float plane for the level-0 collapse. The collapsed result out[k] has 3 planes.
//
//   k_pyr_down_roll    cv::pyrDown, level k -> k+1 of one plane   OCV imgproc/src/pyramids.cpp:745-900 (+344-402, 503-521)
//   k_pyr_down0_roll   level 0 -> 1, one warp per role (the six colour planes of the two images | the mask)
//   k_blend_coarsest   resultSmallest                             reference src/blend.hpp:68-69
//   k_collapse_tma     lap = G - pyrUp(G_coarse) for both images, per-level blend, and out = pyrUp(out_coarse) + blended,
//                      one warp per colour channel fed by a TMA producer warp
//                                                                 reference src/blend.hpp:45-77; pyramids.cpp:903-1005
//   k_collapse_roll    the same on levels without tensor maps (too small to have an interior tile)
//   k_pyramid_tail     the small levels of the pyramid, down and back up, in one CTA per frame
//
// Design (B200: the path is bound by instruction issue, not by HBM, see DESIGN.md).
// A thread owns a few adjacent output columns and walks down a run of rows; the separable filters keep their row-pass
// results in a register window that slides with the walk, so every source row is filtered horizontally once per
// thread column, and the loads of the next step are issued before the current step is computed (software pipeline).
// Global loads are laid out so that a warp instruction reads contiguous 16-byte pieces; taps shared with the
// neighbouring lanes travel by warp shuffle. Work that shares source pixels but not arithmetic (the colour channels / the two images / the mask)
// is split across the warps of a CTA ("roles") so that the sliding windows stay small and the shared loads hit L1.
// Interior tiles and border tiles run different bodies: an INTERIOR one (no border logic at all, vector loads or rows
// staged in shared memory by TMA, the reference's vector-body association everywhere) and a generic one
// (cv::borderInterpolate on every tap, association selected per element, any size down to 1x1); a warp picks one with a
// single uniform branch.
//
// Bit-exactness: OpenCV's SSE-baseline vector bodies associate the 5-tap sums differently from the scalar code
// that handles row borders and loop tails, so the association is selected per element position exactly as the
// reference loops do (DownSel below); all adds and multiplies are individually rounded (no FMA contraction).
#include "common.cuh"
#include "kernels.cuh"
#include "pixel_ops.cuh"
#include "tma.cuh"

namespace poppy {

namespace {

constexpr unsigned FULL = 0xffffffffu;

// Loads of the generic (border / tiny-level) bodies. CG = false: read-only path (data written by an earlier kernel).
// CG = true: ld.global.ca instead of the non-coherent ld.global.nc - for k_pyramid_tail, where one CTA reads what it wrote
// a level earlier (a CTA lives on one SM, whose L1 sees the CTA's own stores; the taps of a tiny level then hit L1).
template <bool CG, class T> __device__ __forceinline__ T ld_in(const T* p) { return CG ? __ldca(p) : __ldg(p); }

// horizontal 1-4-6-4-1, vector-body association: r2*6 + ((r1+r3)*4 + (r0+r4))
__device__ __forceinline__ float h5_vec(float t0, float t1, float t2, float t3, float t4) {
    return __fadd_rn(__fmul_rn(t2, 6.f), __fadd_rn(__fmul_rn(__fadd_rn(t1, t3), 4.f), __fadd_rn(t0, t4)));
}
// scalar association: ((r2*6 + (r1+r3)*4) + r0) + r4
__device__ __forceinline__ float h5_sca(float t0, float t1, float t2, float t3, float t4) {
    return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(t2, 6.f), __fmul_rn(__fadd_rn(t1, t3), 4.f)), t0), t4);
}
// vertical, vector body: ((r1+r3+r2)*4 + (r0+r4+(r2+r2))) * 1/256
__device__ __forceinline__ float v5_vec(float r0, float r1, float r2, float r3, float r4) {
    const float a = __fmul_rn(__fadd_rn(__fadd_rn(r1, r3), r2), 4.f);
    const float b = __fadd_rn(__fadd_rn(r0, r4), __fadd_rn(r2, r2));
    return __fmul_rn(__fadd_rn(a, b), 1.f / 256);
}
__device__ __forceinline__ float v5_sca(float r0, float r1, float r2, float r3, float r4) {
    return __fmul_rn(h5_sca(r0, r1, r2, r3, r4), 1.f / 256);
}

// Which output columns the reference's vector bodies produce (pyramids.cpp:380-402 cn=3, 344-360 cn=1, 503-521);
// all other positions come from the scalar loops.
struct DownSel {
    int width0, h1_end, v_end3, v_end1;
    __device__ DownSel(int sw, int dw) {
        width0 = min((sw - 3) / 2 + 1, dw);
        const int k1 = width0 >= 5 ? (width0 - 5) / 4 + 1 : 0;
        h1_end = 1 + 4 * k1;
        v_end3 = (dw * 3) & ~3;
        v_end1 = dw & ~3;
    }
    __device__ __forceinline__ bool h3(int x) const { return x >= 1 && x <= width0 - 2; }
    __device__ __forceinline__ bool h1(int x) const { return x >= 1 && x < h1_end; }
    __device__ __forceinline__ bool v3(int x, int ch) const { return 3 * x + ch < v_end3; }
    __device__ __forceinline__ bool v1(int x) const { return x < v_end1; }
};

constexpr int DN_R = 16;          // output rows per warp of the pyrDown kernels

// Per-thread association flags of 4 adjacent output columns x..x+3 of one plane kind (bit i: vector-body association).
struct DownFlags { unsigned h, v; };
__device__ __forceinline__ DownFlags down_flags(const DownSel& sel, int x, bool three, int ch) {
    DownFlags f{0u, 0u};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (three ? sel.h3(x + i) : sel.h1(x + i)) f.h |= 1u << i;
        if (three ? sel.v3(x + i, ch) : sel.v1(x + i)) f.v |= 1u << i;
    }
    return f;
}
// Can this thread (output columns x..x+3 of a source row of sw pixels) run the INTERIOR body?
__device__ __forceinline__ bool down_lane_interior(int x, int sw, int dw, DownFlags f) {
    return x + 3 < dw && 2 * x - 2 >= 0 && 2 * x + 8 <= sw - 1 && f.h == 15u && f.v == 15u;
}

// row pass of 4 adjacent outputs from the 11 taps s[2x-2 .. 2x+8]
template <bool INTERIOR>
__device__ __forceinline__ void h5x4(const float (&t)[11], unsigned hflags, float (&o)[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
        o[i] = (INTERIOR || ((hflags >> i) & 1u)) ? h5_vec(t[2 * i], t[2 * i + 1], t[2 * i + 2], t[2 * i + 3], t[2 * i + 4])
                                                  : h5_sca(t[2 * i], t[2 * i + 1], t[2 * i + 2], t[2 * i + 3], t[2 * i + 4]);
}
template <bool INTERIOR>
__device__ __forceinline__ float4 v5x4(const float (&r0)[4], const float (&r1)[4], const float (&r2)[4], const float (&r3)[4],
                                       const float (&r4)[4], unsigned vflags) {
    float o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
        o[i] = (INTERIOR || ((vflags >> i) & 1u)) ? v5_vec(r0[i], r1[i], r2[i], r3[i], r4[i]) : v5_sca(r0[i], r1[i], r2[i], r3[i], r4[i]);
    return make_float4(o[0], o[1], o[2], o[3]);
}

// ---- level k -> k+1, float planes -----------------------------------------------------------------------------------
// A warp covers 128 output columns as two chunks of 64; in chunk j lane l produces outputs xo = X0 + 64j + 2l, xo+1.
// Its own four source values s[2xo .. 2xo+3] are one perfectly coalesced 128-bit load (lane stride 16 bytes); the taps it
// shares with its neighbours (s[2xo-2], s[2xo-1] from lane l-1, s[2xo+4] from lane l+1) arrive by shuffle, and the two
// lanes at the chunk ends fetch theirs with one predicated load each.
struct DownRaw { float4 own; float2 left; float right; };      // left/right: only lane 0 / lane 31 load them

template <bool INTERIOR>
__device__ __forceinline__ void down_load(const float* __restrict__ plane, int spitch, int sh, int iy, int xo, int lane,
                                          DownRaw& r) {
    if (INTERIOR) {
        const float* __restrict__ p = plane + (size_t)iy * spitch + 2 * xo;
        r.own = __ldg(reinterpret_cast<const float4*>(p));
        if (lane == 0) r.left = __ldg(reinterpret_cast<const float2*>(p - 2));
        if (lane == 31) r.right = __ldg(p + 4);
    }
}

// row pass of outputs xo, xo+1 of source row iy
template <bool INTERIOR, bool CG = false>
__device__ __forceinline__ float2 down_rowpass(const float* __restrict__ plane, int spitch, int sw, int sh, int iy, int xo,
                                               int lane, const DownRaw& r, bool va, bool vb, bool has_b) {
    if (INTERIOR) {
        float l2 = __shfl_up_sync(FULL, r.own.z, 1), l1 = __shfl_up_sync(FULL, r.own.w, 1);
        float r0 = __shfl_down_sync(FULL, r.own.x, 1);
        if (lane == 0) { l2 = r.left.x; l1 = r.left.y; }
        if (lane == 31) r0 = r.right;
        return make_float2(h5_vec(l2, l1, r.own.x, r.own.y, r.own.z), h5_vec(r.own.x, r.own.y, r.own.z, r.own.w, r0));
    } else {
        const float* __restrict__ row = plane + (size_t)reflect101(iy, sh) * spitch;
        float t[5];
#pragma unroll
        for (int j = 0; j < 5; ++j) t[j] = ld_in<CG>(row + reflect101(2 * xo - 2 + j, sw));
        float2 o;
        o.x = va ? h5_vec(t[0], t[1], t[2], t[3], t[4]) : h5_sca(t[0], t[1], t[2], t[3], t[4]);
        o.y = 0.f;
        if (has_b) {
#pragma unroll
            for (int j = 0; j < 5; ++j) t[j] = ld_in<CG>(row + reflect101(2 * xo + j, sw));
            o.y = vb ? h5_vec(t[0], t[1], t[2], t[3], t[4]) : h5_sca(t[0], t[1], t[2], t[3], t[4]);
        }
        return o;
    }
}

// One chunk (64 output columns) x DN_R output rows of one plane. Flags: bit 0/1 = vector-body association of the row
// pass at xo / xo+1, bit 2/3 = of the column pass.
template <bool INTERIOR, int R = DN_R, bool CG = false>
__device__ __forceinline__ void down_chunk_f32(const float* __restrict__ sp, int sw, int sh, int spitch, float* __restrict__ dp,
                                               int dw, int dh, int dpitch, int xo, int y0, int lane, unsigned flags) {
    const bool ha = flags & 1u, hb = flags & 2u, va = flags & 4u, vb = flags & 8u, has_b = INTERIOR || xo + 1 < dw;
    float2 h0, h1, h2, h3, h4;
    DownRaw ra, rb;
    down_load<INTERIOR>(sp, spitch, sh, 2 * y0 - 2, xo, lane, ra);
    down_load<INTERIOR>(sp, spitch, sh, 2 * y0 - 1, xo, lane, rb);
    h0 = down_rowpass<INTERIOR, CG>(sp, spitch, sw, sh, 2 * y0 - 2, xo, lane, ra, ha, hb, has_b);
    h1 = down_rowpass<INTERIOR, CG>(sp, spitch, sw, sh, 2 * y0 - 1, xo, lane, rb, ha, hb, has_b);
    down_load<INTERIOR>(sp, spitch, sh, 2 * y0, xo, lane, ra);
    h2 = down_rowpass<INTERIOR, CG>(sp, spitch, sw, sh, 2 * y0, xo, lane, ra, ha, hb, has_b);
    // software pipeline: the two source rows of output row y+1 are requested before output row y is computed
    down_load<INTERIOR>(sp, spitch, sh, 2 * y0 + 1, xo, lane, ra);
    down_load<INTERIOR>(sp, spitch, sh, 2 * y0 + 2, xo, lane, rb);
#pragma unroll 1
    for (int k = 0; k < R; ++k) {
        const int y = y0 + k;
        if (!INTERIOR && y >= dh) break;
        h3 = down_rowpass<INTERIOR, CG>(sp, spitch, sw, sh, 2 * y + 1, xo, lane, ra, ha, hb, has_b);
        h4 = down_rowpass<INTERIOR, CG>(sp, spitch, sw, sh, 2 * y + 2, xo, lane, rb, ha, hb, has_b);
        if (k + 1 < R) {
            down_load<INTERIOR>(sp, spitch, sh, 2 * y + 3, xo, lane, ra);
            down_load<INTERIOR>(sp, spitch, sh, 2 * y + 4, xo, lane, rb);
        }
        float2 o;
        o.x = (INTERIOR || va) ? v5_vec(h0.x, h1.x, h2.x, h3.x, h4.x) : v5_sca(h0.x, h1.x, h2.x, h3.x, h4.x);
        o.y = (INTERIOR || vb) ? v5_vec(h0.y, h1.y, h2.y, h3.y, h4.y) : v5_sca(h0.y, h1.y, h2.y, h3.y, h4.y);
        *reinterpret_cast<float2*>(dp + (size_t)y * dpitch + xo) = o;
        h0 = h2; h1 = h3; h2 = h4;
    }
}

__device__ __forceinline__ unsigned down_pair_flags(const DownSel& sel, int xo, bool three, int ch) {
    unsigned f = 0;
    if (three ? sel.h3(xo) : sel.h1(xo)) f |= 1u;
    if (three ? sel.h3(xo + 1) : sel.h1(xo + 1)) f |= 2u;
    if (three ? sel.v3(xo, ch) : sel.v1(xo)) f |= 4u;
    if (three ? sel.v3(xo + 1, ch) : sel.v1(xo + 1)) f |= 8u;
    return f;
}
__device__ __forceinline__ bool down_pair_interior(int xo, int sw, int dw, unsigned flags) {
    return xo + 1 < dw && 2 * xo - 2 >= 0 && 2 * xo + 4 <= sw - 1 && flags == 15u;
}

}  // namespace

// block (32, 4); grid (ceil(dw/128), ceil(dh/(4 R)), frames * 7): blockIdx.z is the plane job f*7+p, whose planes start
// at job * stride in both levels. Warp wy of a CTA produces output rows (blockIdx.y*4 + wy)*R .. +R-1. R = 16 on the large
// levels (every source row is filtered once per 16 output rows); the small levels, whose grids would not fill the GPU and
// whose walks are pure latency, use R = 4: four times the warps, each a quarter as long.
template <int R>
__global__ void __launch_bounds__(128, 12)      // 40 registers: the walk is latency-bound, residency pays more than the few spills
k_pyr_down_roll(const float* __restrict__ src, int sw, int sh, int spitch, size_t sstride, float* __restrict__ dst, int dw,
                int dh, int dpitch, size_t dstride) {
    const int job = blockIdx.z, p = job % 7, lane = threadIdx.x;
    const int y0 = (blockIdx.y * 4 + threadIdx.y) * R;
    if (y0 >= dh) return;
    const float* __restrict__ sp = src + (size_t)job * sstride;
    float* __restrict__ dp = dst + (size_t)job * dstride;
    const DownSel sel(sw, dw);
    const bool rows_in = 2 * y0 - 2 >= 0 && 2 * (y0 + R - 1) + 2 <= sh - 1 && y0 + R <= dh;
#pragma unroll 1
    for (int j = 0; j < 2; ++j) {
        const int xo = blockIdx.x * 128 + 64 * j + 2 * lane;
        const unsigned flags = down_pair_flags(sel, xo, p < 6, p % 3);
        if (__all_sync(FULL, rows_in && down_pair_interior(xo, sw, dw, flags)))
            down_chunk_f32<true, R>(sp, sw, sh, spitch, dp, dw, dh, dpitch, xo, y0, lane, flags);
        else if (xo < dw)
            down_chunk_f32<false, R>(sp, sw, sh, spitch, dp, dw, dh, dpitch, xo, y0, lane, flags);
    }
}

// ---- level 0 -> 1 -----------------------------------------------------------------------------------------------------
namespace {

// the 11 taps s[2x-2 .. 2x+8] of the thread's 4 outputs from source row iy of level 0 (T = uint32_t: packed BGRX words of
// one warped image; T = float: the mask basis)
template <class T>
__device__ __forceinline__ void down0_taps(const T* __restrict__ plane, int spitch, int sw, int sh, int iy, int x, T (&t)[11]) {
    const T* __restrict__ row = plane + (size_t)reflect101(iy, sh) * spitch;
#pragma unroll
    for (int j = 0; j < 11; ++j) t[j] = __ldg(row + reflect101(2 * x - 2 + j, sw));
}

// roles 0 / 1, border tiles: the three colour planes of one warped image (`words`: its packed BGRX plane). fl.h: row-pass
// flags; fl.v: column-pass flags of the three channels, 4 bits each.
__device__ __forceinline__ void down0_body_img(const uint32_t* __restrict__ words, int wpitch, int sw, int sh,
                                               float* __restrict__ dp /* first of the image's 3 planes */, size_t dstride, int dh,
                                               int dpitch, int x, int y0, DownFlags fl) {
    float h[3][5][4];
    auto rowpass = [&](int iy, int slot) {
        uint32_t wd[11];
        down0_taps(words, wpitch, sw, sh, iy, x, wd);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float t[11];
#pragma unroll
            for (int j = 0; j < 11; ++j) t[j] = unit_from_byte(wd[j], c);
            h5x4<false>(t, fl.h, h[c][slot]);
        }
    };
    rowpass(2 * y0 - 2, 0);
    rowpass(2 * y0 - 1, 1);
    rowpass(2 * y0, 2);
#pragma unroll 1
    for (int k = 0; k < DN_R; ++k) {
        const int y = y0 + k;
        if (y >= dh) break;
        rowpass(2 * y + 1, 3);
        rowpass(2 * y + 2, 4);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            *reinterpret_cast<float4*>(dp + (size_t)c * dstride + (size_t)y * dpitch + x) =
                v5x4<false>(h[c][0], h[c][1], h[c][2], h[c][3], h[c][4], (fl.v >> (4 * c)) & 15u);
#pragma unroll
            for (int i = 0; i < 4; ++i) { h[c][0][i] = h[c][2][i]; h[c][1][i] = h[c][3][i]; h[c][2][i] = h[c][4][i]; }
        }
    }
}

// role 2, border tiles: the blend mask — evaluates lbmask from the mask basis, keeps it as the level-0 mask plane (own
// rows and columns only) and reduces it to level 1
__device__ __forceinline__ void down0_body_mask(const float* __restrict__ basis, int bpitch, double alpha, double beta, int sw,
                                                int sh, float* __restrict__ mask0, float* __restrict__ dp, int dh, int dpitch,
                                                int x, int y0, DownFlags fl) {
    float h[5][4];
    auto rowpass = [&](int iy, int slot) {
        float t[11];
        down0_taps(basis, bpitch, sw, sh, iy, x, t);
#pragma unroll
        for (int j = 0; j < 11; ++j) t[j] = blend_mask(t[j], alpha, beta);
        // level-0 mask plane: this thread owns source columns 2x .. 2x+7 of the source rows 2*y0 .. 2*y0 + 2*DN_R - 1
        if (iy >= 2 * y0 && iy < 2 * y0 + 2 * DN_R && iy < sh) {
            float* __restrict__ m = mask0 + (size_t)iy * bpitch + 2 * x;
            if (2 * x + 7 < sw) {
                *reinterpret_cast<float4*>(m) = make_float4(t[2], t[3], t[4], t[5]);
                *reinterpret_cast<float4*>(m + 4) = make_float4(t[6], t[7], t[8], t[9]);
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (2 * x + j < sw) m[j] = t[2 + j];
            }
        }
        h5x4<false>(t, fl.h, h[slot]);
    };
    rowpass(2 * y0 - 2, 0);
    rowpass(2 * y0 - 1, 1);
    rowpass(2 * y0, 2);
#pragma unroll 1
    for (int k = 0; k < DN_R; ++k) {
        const int y = y0 + k;
        if (y >= dh) break;
        rowpass(2 * y + 1, 3);
        rowpass(2 * y + 2, 4);
        *reinterpret_cast<float4*>(dp + (size_t)y * dpitch + x) = v5x4<false>(h[0], h[1], h[2], h[3], h[4], fl.v);
#pragma unroll
        for (int i = 0; i < 4; ++i) { h[0][i] = h[2][i]; h[1][i] = h[3][i]; h[2][i] = h[4][i]; }
    }
}


// ---- TMA bulk-copy staging of the level 0 -> 1 kernel ----------------------------------------------------------------
// An INTERIOR walk that keeps its loads in registers is bound by memory-level parallelism (one step ahead, ~2 KB in
// flight per warp). Instead every role warp owns a ring of D0_NS source-row segments in shared memory that its lane 0 keeps
// full with cp.async.bulk (the 1-D form of TMA: one instruction per 1056-byte row segment, completion signalled on an
// mbarrier), so ~8 KB per warp are in flight without holding a single register, and the walk itself only issues
// shared-memory loads. A ring is private to its warp: the only synchronisation is the stage's mbarrier (data landed)
// and a __syncwarp() + fence.proxy.async before a consumed stage is refilled.
constexpr int D0_NS = 8;                   // ring depth in source rows
constexpr int D0_SEG = 264;                // elements per staged segment: source columns 2*X0 - 4 .. 2*X0 + 259
constexpr int D0_ROWS = 2 * DN_R + 3;      // source rows 2*y0 - 2 .. 2*y0 + 2*DN_R of one walk
struct __align__(128) Down0Ring {
    uint32_t row[D0_NS][D0_SEG];
    unsigned long long bar[D0_NS];
};
constexpr size_t D0_SMEM = sizeof(Down0Ring) * 3;

// Producer side of one warp's ring: `seg0` points at element (row 2*y0 - 2, column 2*X0 - 4) of the role's source plane.
template <class T>
struct Down0Feed {
    Down0Ring* ring; const T* seg0; int pitch, lane;
    __device__ __forceinline__ void issue(int r) const {           // lane 0 only
        unsigned long long* bar = &ring->bar[r % D0_NS];
        mbar_expect_tx(bar, D0_SEG * 4);
        bulk_g2s(ring->row[r % D0_NS], seg0 + (size_t)r * pitch, D0_SEG * 4, bar);
    }
    __device__ __forceinline__ void start() const {
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < D0_NS; ++i) mbar_init(&ring->bar[i], 1);
            asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
#pragma unroll
            for (int r = 0; r < D0_NS; ++r) issue(r);
        }
        __syncwarp();
    }
    // the 11 taps s[2x-2 .. 2x+8] of this lane's 4 outputs from staged row r (relative to 2*y0 - 2)
    __device__ __forceinline__ void taps(int r, T (&t)[11]) const {
        mbar_wait(&ring->bar[r % D0_NS], (unsigned)(r / D0_NS) & 1u);
        const uint32_t* seg = ring->row[r % D0_NS] + 8 * lane;
        const uint2 l = *reinterpret_cast<const uint2*>(seg + 2);
        const uint4 a = *reinterpret_cast<const uint4*>(seg + 4), b = *reinterpret_cast<const uint4*>(seg + 8);
        const uint32_t r0 = seg[12];
        const uint32_t w[11] = {l.x, l.y, a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, r0};
#pragma unroll
        for (int j = 0; j < 11; ++j) t[j] = *reinterpret_cast<const T*>(&w[j]);
    }
    // rows r0 .. r0 + n - 1 have been consumed by every lane: refill their stages with the rows D0_NS further down
    __device__ __forceinline__ void refill(int r0, int n) const {
        __syncwarp();
        // The stage was read through the generic proxy and is about to be written through the async proxy (TMA): without
        // this cross-proxy fence the refill can overtake the reads (seen on B200 as rare +-1 LSB differences in the first
        // frames of a chunk when two render lanes overlap; tools/stress_determinism.py).
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        if (lane == 0) {
            for (int r = r0 + D0_NS; r < r0 + n + D0_NS; ++r)
                if (r < D0_ROWS) issue(r);
        }
    }
};

// roles 0 / 1, INTERIOR tiles, staged source
__device__ __forceinline__ void down0_bulk_img(const Down0Feed<uint32_t>& F, float* __restrict__ dp, size_t dstride, int dpitch,
                                               int x, int y0) {
    float h[3][5][4];
    auto rowpass = [&](int r, int slot) {
        uint32_t wd[11];
        F.taps(r, wd);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float t[11];
#pragma unroll
            for (int j = 0; j < 11; ++j) t[j] = unit_from_byte(wd[j], c);
            h5x4<true>(t, 15u, h[c][slot]);
        }
    };
    F.start();
    rowpass(0, 0);
    rowpass(1, 1);
    rowpass(2, 2);
    F.refill(0, 3);
#pragma unroll 1
    for (int k = 0; k < DN_R; ++k) {
        const int y = y0 + k;
        rowpass(2 * k + 3, 3);
        rowpass(2 * k + 4, 4);
        F.refill(2 * k + 3, 2);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            *reinterpret_cast<float4*>(dp + (size_t)c * dstride + (size_t)y * dpitch + x) =
                v5x4<true>(h[c][0], h[c][1], h[c][2], h[c][3], h[c][4], 15u);
#pragma unroll
            for (int i = 0; i < 4; ++i) { h[c][0][i] = h[c][2][i]; h[c][1][i] = h[c][3][i]; h[c][2][i] = h[c][4][i]; }
        }
    }
}

// role 2, INTERIOR tiles, staged mask basis
__device__ __forceinline__ void down0_bulk_mask(const Down0Feed<float>& F, int bpitch, double alpha, double beta,
                                                float* __restrict__ mask0, float* __restrict__ dp, int dpitch, int x, int y0) {
    float h[5][4];
    auto rowpass = [&](int r, int slot) {
        float t[11];
        F.taps(r, t);
#pragma unroll
        for (int j = 0; j < 11; ++j) t[j] = blend_mask(t[j], alpha, beta);
        if (r >= 2 && r < 2 + 2 * DN_R) {          // source rows 2*y0 .. 2*y0 + 2*DN_R - 1: this warp owns their level-0 mask
            float* __restrict__ m = mask0 + (size_t)(2 * y0 - 2 + r) * bpitch + 2 * x;
            *reinterpret_cast<float4*>(m) = make_float4(t[2], t[3], t[4], t[5]);
            *reinterpret_cast<float4*>(m + 4) = make_float4(t[6], t[7], t[8], t[9]);
        }
        h5x4<true>(t, 15u, h[slot]);
    };
    F.start();
    rowpass(0, 0);
    rowpass(1, 1);
    rowpass(2, 2);
    F.refill(0, 3);
#pragma unroll 1
    for (int k = 0; k < DN_R; ++k) {
        const int y = y0 + k;
        rowpass(2 * k + 3, 3);
        rowpass(2 * k + 4, 4);
        F.refill(2 * k + 3, 2);
        *reinterpret_cast<float4*>(dp + (size_t)y * dpitch + x) = v5x4<true>(h[0], h[1], h[2], h[3], h[4], 15u);
#pragma unroll
        for (int i = 0; i < 4; ++i) { h[0][i] = h[2][i]; h[1][i] = h[3][i]; h[2][i] = h[4][i]; }
    }
}

}  // namespace

// block (32, 3): three row groups of one role (0: image 1, 1: image 2, 2: mask); grid (ceil(dw/128), ceil(dh/48), 3 * frames).
// warped: per frame two planes of packed BGRX words (image 1, image 2), rows wpitch words apart, wstride words per
// plane. mask0: per-frame level-0 mask planes (rows bpitch floats apart, m0stride floats per frame) written here for the
// level-0 collapse. Interior tiles stage their source rows through a Down0Feed ring, border tiles run the generic bodies.
// SEG: frame f's mask basis is its segment's, seg[f].basis (same pitch; every basis starts 128-byte aligned).
template <bool SEG>
__device__ __forceinline__ void
pyr_down0_body(const uint32_t* __restrict__ warped, int wpitch, size_t wstride, const float* __restrict__ basis, int bpitch,
               const SegFrame* __restrict__ seg, const FrameParams* __restrict__ fp, int sw, int sh, float* __restrict__ mask0,
               size_t m0stride, float* __restrict__ dst, int dw, int dh, int dpitch, size_t dstride) {
    extern __shared__ __align__(128) unsigned char smem_down0[];
    // blockIdx.z = role * frames + f: CTAs that are resident together run the same role, i.e. the same hot loop, which
    // keeps the per-scheduler instruction cache from thrashing between the (large, fully unrolled) role bodies. The three
    // warps of a CTA take three consecutive row groups.
    const int frames = gridDim.z / 3, role = blockIdx.z / frames, f = blockIdx.z - role * frames, lane = threadIdx.x;
    const int X0 = blockIdx.x * 128, x = X0 + 4 * lane, y0 = (blockIdx.y * 3 + threadIdx.y) * DN_R;
    if (y0 >= dh) return;
    const int ring_slot = threadIdx.y;
    const DownSel sel(sw, dw);
    const bool rows_in = 2 * y0 - 2 >= 0 && 2 * (y0 + DN_R - 1) + 2 <= sh - 1 && y0 + DN_R <= dh;
    float* __restrict__ dframe = dst + (size_t)f * 7 * dstride;
    if (role < 2) {
        DownFlags fl = down_flags(sel, x, true, 0);
        const unsigned v1 = down_flags(sel, x, true, 1).v, v2 = down_flags(sel, x, true, 2).v;
        const bool lane_in = down_lane_interior(x, sw, dw, fl) && v1 == 15u && v2 == 15u;
        fl.v |= (v1 << 4) | (v2 << 8);
        const uint32_t* __restrict__ words = warped + ((size_t)f * 2 + role) * wstride;
        const bool interior = __all_sync(FULL, rows_in && lane_in) && (2 * X0 - 4 >= 0 && 2 * X0 - 4 + D0_SEG <= wpitch);
        if (interior) {
            const Down0Feed<uint32_t> F{reinterpret_cast<Down0Ring*>(smem_down0) + ring_slot,
                                        words + (size_t)(2 * y0 - 2) * wpitch + 2 * X0 - 4, wpitch, lane};
            down0_bulk_img(F, dframe + (size_t)3 * role * dstride, dstride, dpitch, x, y0);
        } else if (x < dw) {
            down0_body_img(words, wpitch, sw, sh, dframe + (size_t)3 * role * dstride, dstride, dh, dpitch, x, y0, fl);
        }
    } else {
        const DownFlags fl = down_flags(sel, x, false, 0);
        const double alpha = fp[f].mask_alpha, beta = fp[f].mask_beta;
        if (SEG) basis = seg[f].basis;
        float* __restrict__ m0 = mask0 + (size_t)f * m0stride;
        const bool interior = __all_sync(FULL, rows_in && down_lane_interior(x, sw, dw, fl)) &&
                              (2 * X0 - 4 >= 0 && 2 * X0 - 4 + D0_SEG <= bpitch);
        if (interior) {
            const Down0Feed<float> F{reinterpret_cast<Down0Ring*>(smem_down0) + ring_slot,
                                     basis + (size_t)(2 * y0 - 2) * bpitch + 2 * X0 - 4, bpitch, lane};
            down0_bulk_mask(F, bpitch, alpha, beta, m0, dframe + 6 * dstride, dpitch, x, y0);
        } else if (x < dw) {
            down0_body_mask(basis, bpitch, alpha, beta, sw, sh, m0, dframe + 6 * dstride, dh, dpitch, x, y0, fl);
        }
    }
}

__global__ void __launch_bounds__(96)
k_pyr_down0_roll(const uint32_t* __restrict__ warped, int wpitch, size_t wstride, const float* __restrict__ basis, int bpitch,
                 const FrameParams* __restrict__ fp, int sw, int sh, float* __restrict__ mask0, size_t m0stride,
                 float* __restrict__ dst, int dw, int dh, int dpitch, size_t dstride) {
    pyr_down0_body<false>(warped, wpitch, wstride, basis, bpitch, nullptr, fp, sw, sh, mask0, m0stride, dst, dw, dh, dpitch, dstride);
}

__global__ void __launch_bounds__(96)
k_pyr_down0_roll_seg(const uint32_t* __restrict__ warped, int wpitch, size_t wstride, const SegFrame* __restrict__ seg, int bpitch,
                     const FrameParams* __restrict__ fp, int sw, int sh, float* __restrict__ mask0, size_t m0stride,
                     float* __restrict__ dst, int dw, int dh, int dpitch, size_t dstride) {
    pyr_down0_body<true>(warped, wpitch, wstride, nullptr, bpitch, seg, fp, sw, sh, mask0, m0stride, dst, dw, dh, dpitch, dstride);
}

// block 256; grid (ceil(w*h/256), frames)
__global__ void k_blend_coarsest(const float* __restrict__ g, int w, int h, int pitch, size_t stride,
                                 float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, f = blockIdx.y;
    if (i >= w * h) return;
    const size_t o = (size_t)(i / w) * pitch + (i % w);
    const float* gf = g + (size_t)f * 7 * stride + o;
    const float m = gf[6 * stride], anti = __fsub_rn(1.0f, m);
#pragma unroll
    for (int c = 0; c < 3; ++c)
        out[((size_t)f * 3 + c) * stride + o] =
            __fadd_rn(__fmul_rn(gf[(size_t)c * stride], m), __fmul_rn(gf[(size_t)(3 + c) * stride], anti));
}

// ---- collapse ---------------------------------------------------------------------------------------------------------
namespace {

constexpr int CL_R = 16;           // coarse rows per warp of the collapse kernel (32 fine rows x 128 fine columns)

// horizontal pass of cv::pyrUp at fine column x of one coarse row of n pixels (pyramids.cpp:945-978)
template <bool CG = false>
__device__ __forceinline__ float up_h(const float* __restrict__ row, int n, int x) {
    const int sx = x >> 1;
    if (n == 1) return __fmul_rn(ld_in<CG>(row), 8.f);
    if (x & 1) {
        if (sx == n - 1) return __fmul_rn(ld_in<CG>(row + n - 1), 8.f);
        return __fmul_rn(__fadd_rn(ld_in<CG>(row + sx), ld_in<CG>(row + sx + 1)), 4.f);
    }
    if (sx == 0) return __fadd_rn(__fmul_rn(ld_in<CG>(row), 6.f), __fmul_rn(ld_in<CG>(row + 1), 2.f));
    if (sx == n - 1) return __fadd_rn(ld_in<CG>(row + n - 2), __fmul_rn(ld_in<CG>(row + n - 1), 7.f));
    return __fadd_rn(__fadd_rn(ld_in<CG>(row + sx - 1), __fmul_rn(ld_in<CG>(row + sx), 6.f)), ld_in<CG>(row + sx + 1));
}

// Row pass of cv::pyrUp for the 4 fine columns fx..fx+3 (coarse columns a = fx/2, a+1) of one coarse row, scaled by 1/64.
// Scaling by a power of two is exact and commutes with every rounding of the column pass, so applying it here instead of
// after the column sums (pyramids.cpp:989-991) is bit-identical and saves one multiply per value and fine row.
template <bool INTERIOR, bool CG = false>
__device__ __forceinline__ void up_row(const float* __restrict__ row, int cw, int w, int fx, float (&o)[4]) {
    if (INTERIOR) {
        const float* __restrict__ p = row + (fx >> 1);
        const float cm = __ldg(p - 1);
        const float2 c01 = __ldg(reinterpret_cast<const float2*>(p));
        const float cp = __ldg(p + 2);
        o[0] = __fadd_rn(__fadd_rn(cm, __fmul_rn(c01.x, 6.f)), c01.y);
        o[1] = __fmul_rn(__fadd_rn(c01.x, c01.y), 4.f);
        o[2] = __fadd_rn(__fadd_rn(c01.x, __fmul_rn(c01.y, 6.f)), cp);
        o[3] = __fmul_rn(__fadd_rn(c01.y, cp), 4.f);
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) o[i] = fx + i < w ? up_h<CG>(row, cw, fx + i) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = __fmul_rn(o[i], 1.f / 64);
}

// vertical pass of cv::pyrUp (pyramids.cpp:929-993) on pre-scaled row-pass values: even fine row (r0 + 6 r1) + r2, odd fine
// row (r1 + r2) * 4; then out = up_o + ((gl - up_l) * m + (gr - up_r) * (1 - m))   (blend.hpp:52-53,70-72,62-63) - both in the
// column-pair forms below.

// ---- packed fp32 (sm_100 FADD2 / FMUL2 / FFMA2: two individually rounded IEEE operations per issue slot) ------------------
// ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even under --fmad=false (seen with CUDA 12.9), which would
// change the rounding. A product that feeds an addition is therefore issued as fma(a, b, -0.0) with the -0.0 read from
// constant memory (opaque to the compiler): a * b + (-0.0) rounds once to exactly round(a * b), signed zeros included,
// and an FFMA2 cannot be merged with the addition that follows. Multiplications by powers of two are exact, so their
// contraction is harmless and they use FMUL2. a - b is fma(b, -1, a): one rounding of the exact difference.
__constant__ float2 c_negzero2 = {-0.0f, -0.0f};
__device__ __forceinline__ float2 padd(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 psub(float2 a, float2 b) { return __ffma2_rn(b, make_float2(-1.f, -1.f), a); }
__device__ __forceinline__ float2 pmul_rounded(float2 a, float2 b, float2 nz) { return __ffma2_rn(a, b, nz); }
__device__ __forceinline__ float2 pscale(float2 a, float pow2) { return __fmul2_rn(a, make_float2(pow2, pow2)); }
// column-pair forms of up_even / up_odd / blend1
__device__ __forceinline__ float2 up_even2(float2 h0, float2 h1, float2 h2, float2 nz) {
    return padd(padd(h0, pmul_rounded(h1, make_float2(6.f, 6.f), nz)), h2);
}
__device__ __forceinline__ float2 up_odd2(float2 h1, float2 h2) { return pscale(padd(h1, h2), 4.f); }
__device__ __forceinline__ float2 blend2(float2 gl, float2 gr, float2 m, float2 ul, float2 ur, float2 uo, float2 nz) {
    const float2 lap_l = psub(gl, ul), lap_r = psub(gr, ur), anti = psub(make_float2(1.f, 1.f), m);
    return padd(uo, padd(pmul_rounded(lap_l, m, nz), pmul_rounded(lap_r, anti, nz)));
}

struct CollapseArgs {
    // fine level: L0 -> the two warped word planes + level-0 mask plane; else the 7 Gaussian planes
    const uint32_t* w1; const uint32_t* w2; int wpitch;
    const float* mask0; int mpitch;
    const float* gfine; int fpitch; size_t fstride;
    // coarse level
    const float* gc; const float* oc; int cw, ch, cpitch; size_t cstride;
    float* out; int opitch; size_t ostride;
    int w, h;
};

// one step of an interior tile as read from its TMA stage: the coarse taps of a lane's 4 fine columns, the fine values
struct UpRaw { float cm; float2 c01; float cp; };
template <bool L0> struct FineRaw;
template <> struct FineRaw<true> { uint4 a, b; float4 m; };      // 4 px of image 1, of image 2, mask
template <> struct FineRaw<false> { float4 l, r, m; };

__device__ __forceinline__ void up_row_raw(const UpRaw& u, float (&o)[4]) {
    o[0] = __fmul_rn(__fadd_rn(__fadd_rn(u.cm, __fmul_rn(u.c01.x, 6.f)), u.c01.y), 1.f / 64);
    o[1] = __fmul_rn(__fmul_rn(__fadd_rn(u.c01.x, u.c01.y), 4.f), 1.f / 64);
    o[2] = __fmul_rn(__fadd_rn(__fadd_rn(u.c01.x, __fmul_rn(u.c01.y, 6.f)), u.cp), 1.f / 64);
    o[3] = __fmul_rn(__fmul_rn(__fadd_rn(u.c01.y, u.cp), 4.f), 1.f / 64);
}

template <bool L0>
__device__ __forceinline__ void fine_load(const CollapseArgs& A, int c, int fy, int fx, FineRaw<L0>& r);
template <>
__device__ __forceinline__ void fine_load<true>(const CollapseArgs& A, int c, int fy, int fx, FineRaw<true>& r) {
    const size_t o = (size_t)fy * A.wpitch + fx;
    r.a = __ldg(reinterpret_cast<const uint4*>(A.w1 + o));
    r.b = __ldg(reinterpret_cast<const uint4*>(A.w2 + o));
    r.m = __ldg(reinterpret_cast<const float4*>(A.mask0 + (size_t)fy * A.mpitch + fx));
}
template <>
__device__ __forceinline__ void fine_load<false>(const CollapseArgs& A, int c, int fy, int fx, FineRaw<false>& r) {
    const float* __restrict__ gp = A.gfine + (size_t)fy * A.fpitch + fx;
    r.l = __ldg(reinterpret_cast<const float4*>(gp + (size_t)c * A.fstride));
    r.r = __ldg(reinterpret_cast<const float4*>(gp + (size_t)(3 + c) * A.fstride));
    r.m = __ldg(reinterpret_cast<const float4*>(gp + (size_t)6 * A.fstride));
}
// the same through the coherent path (k_pyramid_tail)
__device__ __forceinline__ void fine_load_cg(const CollapseArgs& A, int c, int fy, int fx, FineRaw<false>& r) {
    const float* gp = A.gfine + (size_t)fy * A.fpitch + fx;
    r.l = __ldca(reinterpret_cast<const float4*>(gp + (size_t)c * A.fstride));
    r.r = __ldca(reinterpret_cast<const float4*>(gp + (size_t)(3 + c) * A.fstride));
    r.m = __ldca(reinterpret_cast<const float4*>(gp + (size_t)6 * A.fstride));
}
__device__ __forceinline__ void fine_unpack(const FineRaw<true>& r, int c, float (&gl)[4], float (&gr)[4], float (&mk)[4]) {
    gl[0] = unit_from_byte(r.a.x, c); gl[1] = unit_from_byte(r.a.y, c); gl[2] = unit_from_byte(r.a.z, c); gl[3] = unit_from_byte(r.a.w, c);
    gr[0] = unit_from_byte(r.b.x, c); gr[1] = unit_from_byte(r.b.y, c); gr[2] = unit_from_byte(r.b.z, c); gr[3] = unit_from_byte(r.b.w, c);
    mk[0] = r.m.x; mk[1] = r.m.y; mk[2] = r.m.z; mk[3] = r.m.w;
}
__device__ __forceinline__ void fine_unpack(const FineRaw<false>& r, int c, float (&gl)[4], float (&gr)[4], float (&mk)[4]) {
    gl[0] = r.l.x; gl[1] = r.l.y; gl[2] = r.l.z; gl[3] = r.l.w;
    gr[0] = r.r.x; gr[1] = r.r.y; gr[2] = r.r.z; gr[3] = r.r.w;
    mk[0] = r.m.x; mk[1] = r.m.y; mk[2] = r.m.z; mk[3] = r.m.w;
}

__device__ __forceinline__ void fine_from_rows(float4 a, float4 b, float4 m, FineRaw<true>& f) {
    f.a = make_uint4(__float_as_uint(a.x), __float_as_uint(a.y), __float_as_uint(a.z), __float_as_uint(a.w));
    f.b = make_uint4(__float_as_uint(b.x), __float_as_uint(b.y), __float_as_uint(b.z), __float_as_uint(b.w));
    f.m = m;
}
__device__ __forceinline__ void fine_from_rows(float4 l, float4 r, float4 m, FineRaw<false>& f) { f.l = l; f.r = r; f.m = m; }

// ---- fused 8-bit store of the level-0 collapse ("calm" route of the unsharp stage) -------------------------------------
// unsharp_mask() leaves a pixel untouched unless the 3x3 median of d = x - GaussianBlur(x, sigma 1) reaches norm 0.3
// (src/util.cpp:135-145). With the symmetric 9-tap kernel, d = (I - Bx) x + Bx (I - By) x and
//     (I - Bx) x (p) = - sum_{a>0} w_a [x(p+a) + x(p-a) - 2 x(p)],   |x(p+a) + x(p-a) - 2 x(p)| <= a^2 max |d2x|,
// so |d| <= 0.5 (max |d2x| + max |d2y|) over the pixel's footprint (sum_{a>0} w_a a^2 = 0.499964 <= 0.49997), d2 being
// the unit second differences of x (reflected at the image border like the blur). Where that bound stays below 0.1732 in every channel no
// median can reach the threshold (3 * 0.1732^2 < 0.09) and the frame pixel is exactly cvRound(255 x): neither blur nor
// median have to be evaluated. The level-0 collapse therefore stores the 8-bit frame itself; k_calm_scan
// (kernels_unsharp.cu) bounds the second differences from the stored bytes (|x - byte/255| <= 0.5/255 unless x was clamped,
// which this kernel records per 4x8 block as `excess`), and only the strip chunks that fail the bound run the exact blur +
// median path, which overwrites them (launch_collapse0 + k_unsharp_strip on the flagged tiles).
constexpr float EMIT_EXCESS_TOL = 0.255f;      // |255 x - clamp(255 x)| tolerated in a calm block (0.001 in units of x)
struct EmitCtx {
    uint8_t* frame;            // ring slot of the frame: tight rows of 3 * w bytes
    unsigned char* ex;         // clamp-excess flags of this frame and channel: [ceil(h/8)][ex_pitch] blocks of 4x8 pixels
    int ex_pitch;
    unsigned char* rowbuf;     // shared: [2 step parities][2 rows][384 bytes] interleaved BGR of the CTA's 128 columns
    float excess;              // max |255 x - clamp(255 x)| of the lane's current block
};

// cvRound(255 v) saturated to 8 bits as u8_magic() computes it (byte in the low mantissa bits), also tracking how far v
// lies outside [0, 1]
__device__ __forceinline__ float emit_u8(EmitCtx& E, float v) {
    const float t = __fmul_rn(v, 255.f);
    const float cl = fminf(fmaxf(t, 0.f), 255.f);
    E.excess = fmaxf(E.excess, fabsf(__fsub_rn(t, cl)));
    return __fadd_rn(cl, 12582912.0f);
}
__device__ __forceinline__ void emit_flush(EmitCtx& E, int fy, int fx) {
    E.ex[(size_t)(fy / CALM_BLOCK_H) * E.ex_pitch + fx / CALM_BLOCK_W] = E.excess > EMIT_EXCESS_TOL ? 1 : 0;
    E.excess = 0.f;
}
// INTERIOR tiles of k_collapse_tma (the three channel warps in step, w % 4 == 0): the channel warps interleave their bytes
// in shared memory and every warp stores one contiguous 128-byte third of each 384-byte frame row segment
__device__ __forceinline__ void emit_rows_interior(EmitCtx& E, int k, const float (&e)[4], const float (&o)[4], int c, int lane,
                                                   int w, int fy, int fx0) {
    unsigned char* b = E.rowbuf + (k & 1) * 768;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        b[12 * lane + 3 * i + c] = (unsigned char)(__float_as_uint(emit_u8(E, e[i])) & 255u);
        b[384 + 12 * lane + 3 * i + c] = (unsigned char)(__float_as_uint(emit_u8(E, o[i])) & 255u);
    }
    // one barrier per step: the buffers alternate with the step parity (a named barrier of the three channel warps: the
    // producer warp does not take part)
    asm volatile("bar.sync 1, 96;\n" ::: "memory");
    const uint32_t* bw = reinterpret_cast<const uint32_t*>(b);
    const uint32_t w0 = bw[32 * c + lane], w1 = bw[96 + 32 * c + lane];
    uint32_t* drow = reinterpret_cast<uint32_t*>(E.frame + ((size_t)fy * w + fx0) * 3) + 32 * c + lane;
    drow[0] = w0;
    drow[(size_t)w * 3 / 4] = w1;
    if ((k & 3) == 3) emit_flush(E, fy, fx0 + 4 * lane);
}
// any tile, any lane subset: every lane stores the bytes of its own channel
__device__ __forceinline__ void emit_rows_generic(EmitCtx& E, int k, const float (&e)[4], const float (&o)[4], bool two, int c, int w,
                                                  int fy, int fx) {
    const int n = min(4, w - fx);
    uint8_t* d0 = E.frame + ((size_t)fy * w + fx) * 3 + c;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (i < n) {
            d0[3 * i] = (uint8_t)(__float_as_uint(emit_u8(E, e[i])) & 255u);
            if (two) d0[(size_t)w * 3 + 3 * i] = (uint8_t)(__float_as_uint(emit_u8(E, o[i])) & 255u);
        }
    if ((k & 3) == 3) emit_flush(E, fy, fx);
}

// One warp = one colour channel c of a 128 x 32 fine tile, any tile (cv::borderInterpolate on every tap).
template <bool L0, bool EMIT = false, bool CG = false>
__device__ __forceinline__ void collapse_body(const CollapseArgs& A, int c, int fx, int cy0, EmitCtx* E = nullptr, int R = CL_R) {
    const float* __restrict__ pl = A.gc + (size_t)c * A.cstride;
    const float* __restrict__ pr = A.gc + (size_t)(3 + c) * A.cstride;
    const float* __restrict__ po = A.oc + (size_t)c * A.cstride;
    const float2 nz = c_negzero2;
    float hm[3][4], h0[3][4], hp[3][4];          // row-pass values of coarse rows sy-1, sy, sy+1 for (left, right, out)
    auto coarse_now = [&](int cy, float (&h)[3][4]) {            // load where consumed
        const size_t off = (size_t)cy * A.cpitch;
        up_row<false, CG>(pl + off, A.cw, A.w, fx, h[0]);
        up_row<false, CG>(pr + off, A.cw, A.w, fx, h[1]);
        up_row<false, CG>(po + off, A.cw, A.w, fx, h[2]);
    };
    // borderInterpolate(2(sy-1), 2ch, REFLECT_101)/2: row -1 -> 1 (0 when the level has a single row)
    coarse_now(cy0 >= 1 ? cy0 - 1 : (A.ch > 1 ? 1 : 0), hm);
    coarse_now(cy0, h0);
    float* __restrict__ orow = EMIT ? nullptr : A.out + (size_t)c * A.ostride + (size_t)(2 * cy0) * A.opitch + fx;
    int k_done = 0;
#pragma unroll 1
    for (int k = 0; k < R; ++k) {
        const int sy = cy0 + k, fy = 2 * sy;
        if (fy >= A.h) break;
        k_done = k + 1;
        const bool two = fy + 1 < A.h;
        float gl[2][4], gr[2][4], mk[2][4];
        FineRaw<L0> rf;
        coarse_now(min(sy + 1, A.ch - 1), hp);
        if (CG) fine_load_cg(A, c, fy, fx, reinterpret_cast<FineRaw<false>&>(rf)); else fine_load<L0>(A, c, fy, fx, rf);
        fine_unpack(rf, c, gl[0], gr[0], mk[0]);
        if (two) {
            if (CG) fine_load_cg(A, c, fy + 1, fx, reinterpret_cast<FineRaw<false>&>(rf)); else fine_load<L0>(A, c, fy + 1, fx, rf);
            fine_unpack(rf, c, gl[1], gr[1], mk[1]);
        }
        float e[4], o[4];
#pragma unroll
        for (int i = 0; i < 4; i += 2) {              // two adjacent columns per packed operation
            float2 u[3];
#pragma unroll
            for (int p = 0; p < 3; ++p)
                u[p] = up_even2(make_float2(hm[p][i], hm[p][i + 1]), make_float2(h0[p][i], h0[p][i + 1]),
                                make_float2(hp[p][i], hp[p][i + 1]), nz);
            const float2 ev = blend2(make_float2(gl[0][i], gl[0][i + 1]), make_float2(gr[0][i], gr[0][i + 1]),
                                     make_float2(mk[0][i], mk[0][i + 1]), u[0], u[1], u[2], nz);
            e[i] = ev.x; e[i + 1] = ev.y;
            if (two) {
#pragma unroll
                for (int p = 0; p < 3; ++p)
                    u[p] = up_odd2(make_float2(h0[p][i], h0[p][i + 1]), make_float2(hp[p][i], hp[p][i + 1]));
                const float2 ov = blend2(make_float2(gl[1][i], gl[1][i + 1]), make_float2(gr[1][i], gr[1][i + 1]),
                                         make_float2(mk[1][i], mk[1][i + 1]), u[0], u[1], u[2], nz);
                o[i] = ov.x; o[i + 1] = ov.y;
            }
        }
        if (EMIT) {
            emit_rows_generic(*E, k, e, o, two, c, A.w, fy, fx);
        } else {
            *reinterpret_cast<float4*>(orow) = make_float4(e[0], e[1], e[2], e[3]);
            if (two) *reinterpret_cast<float4*>(orow + A.opitch) = make_float4(o[0], o[1], o[2], o[3]);
            orow += 2 * (size_t)A.opitch;
        }
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
            for (int i = 0; i < 4; ++i) { hm[p][i] = h0[p][i]; h0[p][i] = hp[p][i]; }
    }
    // a block of the min/max table cut short by the image's last rows
    if (EMIT && k_done > 0 && (k_done & 3) != 0) emit_flush(*E, 2 * (cy0 + k_done - 1), fx);
}

}  // namespace

// block (32, 3): warp = colour channel; grid (ceil(w/128), ceil(h/32), frames). The collapse of a level without tensor maps:
// ensure_chunk (poppy_cuda.cu) builds them for every level large enough to have an interior tile, so every tile here takes
// the generic body.
// L0: the fine Gaussian level is the warped 8-bit pair (two word planes per frame, wstride words each) + the level-0
// mask plane written by k_pyr_down0_roll.
// EMIT (level 0 only): instead of the float planes of out[0] the kernel stores the 8-bit frame cvRound(255 out[0]) into the
// frame ring and the per-block clamp-excess flags (see EmitCtx). tile_flags (nullable): per frame and CTA tile, 0 = skip the
// tile (the exact unsharp path only needs out[0] where k_calm_chunks flagged it).
template <bool L0, bool EMIT>
__global__ void __launch_bounds__(96, 8)
k_collapse_roll(const uint32_t* __restrict__ warped, int wpitch, size_t wstride, const float* __restrict__ mask0, int mpitch,
                size_t m0stride, const float* __restrict__ g_fine, int w, int h, int fpitch, size_t fstride,
                const float* __restrict__ g_coarse, const float* __restrict__ out_coarse, int cw, int ch, int cpitch,
                size_t cstride, float* __restrict__ out_fine, int opitch, size_t ostride,
                const unsigned char* __restrict__ tile_flags, const FrameParams* __restrict__ fp, uint8_t* __restrict__ frames_base,
                size_t frame_bytes, unsigned char* __restrict__ ex, int ex_pitch, size_t ex_stride, int R) {
    const int f = blockIdx.z, c = threadIdx.y;
    if (tile_flags && !tile_flags[((size_t)f * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x]) return;
    const int fx = blockIdx.x * 128 + 4 * threadIdx.x, cy0 = blockIdx.y * R;
    if (fx >= w) return;
    CollapseArgs A;
    A.w1 = L0 ? warped + (size_t)f * 2 * wstride : nullptr; A.w2 = L0 ? A.w1 + wstride : nullptr; A.wpitch = wpitch;
    A.mask0 = L0 ? mask0 + (size_t)f * m0stride : nullptr; A.mpitch = mpitch;
    A.gfine = L0 ? nullptr : g_fine + (size_t)f * 7 * fstride; A.fpitch = fpitch; A.fstride = fstride;
    A.gc = g_coarse + (size_t)f * 7 * cstride; A.oc = out_coarse + (size_t)f * 3 * cstride;
    A.cw = cw; A.ch = ch; A.cpitch = cpitch; A.cstride = cstride;
    A.out = EMIT ? nullptr : out_fine + (size_t)f * 3 * ostride; A.opitch = opitch; A.ostride = ostride; A.w = w; A.h = h;
    EmitCtx E;
    if (EMIT) {
        E.frame = frames_base + (size_t)fp[f].dst_slot * frame_bytes;
        E.ex = ex + ((size_t)f * 3 + c) * ex_stride; E.ex_pitch = ex_pitch;
        E.rowbuf = nullptr;        // the generic store writes the frame directly
        E.excess = 0.f;
    }
    collapse_body<L0, EMIT>(A, c, fx, cy0, &E, R);
}

// ---- collapse with a TMA producer warp --------------------------------------------------------------------------------
// Interior tiles of k_collapse_tma: a fourth warp keeps a ring of CT_NS stages full with tensor-map TMA box copies
// (cp.async.bulk.tensor.3d, SASS UTMALDG): per step one box for the two fine rows of the warped pair (both images, 2 KB),
// one for the mask rows, one for the coarse row of the six Gaussian planes and one for the coarse row of the three out
// planes - four instructions per step and CTA instead of 27 per-warp row-segment copies, and the three channel warps
// share the fine data instead of staging it three times. Full/empty mbarriers connect the producer to
// the channel warps; border tiles run the generic body.
constexpr int CT_NS = 3;
template <bool L0> struct CtStage;
template <> struct __align__(128) CtStage<true> {
    uint32_t fine[2][2][128];            // [image][row][column]: box {128, 2, 2} of the warped word planes
    float mask[2][128];                  // box {128, 2, 1} of the level-0 mask
    __align__(128) float gc[6][72];      // box {72, 1, 6}: coarse columns a0-4 .. a0+67 of left B,G,R, right B,G,R
    __align__(128) float oc[3][72];      // box {72, 1, 3} of the coarse out planes
};
template <> struct __align__(128) CtStage<false> {
    float fine[7][2][128];               // box {128, 2, 7} of the fine Gaussian planes
    __align__(128) float gc[6][72];
    __align__(128) float oc[3][72];
};
struct CtBars { unsigned long long full[CT_NS], empty[CT_NS]; };
template <bool L0> __host__ __device__ constexpr unsigned ct_stage_bytes() { return (L0 ? 2 * 2 * 128 * 4 + 2 * 128 * 4 : 7 * 2 * 128 * 4) + 6 * 72 * 4 + 3 * 72 * 4; }
template <bool L0, bool EMIT> constexpr size_t ct_smem() { return CT_NS * sizeof(CtStage<L0>) + 128 + (EMIT ? 2 * 2 * 384 : 0); }

// channel warp c of an interior tile
template <bool L0, bool EMIT>
__device__ __forceinline__ void collapse_consume(const CollapseArgs& A, int c, int fx, int cy0, int lane, const CtStage<L0>* stages,
                                                 CtBars* bars, EmitCtx* E, bool emit_words, int R) {
    const float2 nz = c_negzero2;
    const float* __restrict__ pl = A.gc + (size_t)c * A.cstride;
    const float* __restrict__ pr = A.gc + (size_t)(3 + c) * A.cstride;
    const float* __restrict__ po = A.oc + (size_t)c * A.cstride;
    const int fx0 = fx - 4 * lane;
    float hm[3][4], h0[3][4], hp[3][4];
    {   // coarse rows cy0 - 1 and cy0: loaded directly, once per tile
        const size_t o1 = (size_t)(cy0 - 1) * A.cpitch, o2 = (size_t)cy0 * A.cpitch;
        up_row<true>(pl + o1, A.cw, A.w, fx, hm[0]); up_row<true>(pr + o1, A.cw, A.w, fx, hm[1]); up_row<true>(po + o1, A.cw, A.w, fx, hm[2]);
        up_row<true>(pl + o2, A.cw, A.w, fx, h0[0]); up_row<true>(pr + o2, A.cw, A.w, fx, h0[1]); up_row<true>(po + o2, A.cw, A.w, fx, h0[2]);
    }
    float* __restrict__ orow = EMIT ? nullptr : A.out + (size_t)c * A.ostride + (size_t)(2 * cy0) * A.opitch + fx;
#pragma unroll 1
    for (int k = 0; k < R; ++k) {
        const int s = k % CT_NS, fy = 2 * (cy0 + k);
        mbar_wait(&bars->full[s], (unsigned)(k / CT_NS) & 1u);
        const CtStage<L0>& S = stages[s];
        float gl[2][4], gr[2][4], mk[2][4];
#pragma unroll
        for (int p = 0; p < 3; ++p) {
            const float* seg = (p == 0 ? S.gc[c] : p == 1 ? S.gc[3 + c] : S.oc[c]) + 4 + 2 * lane;      // coarse column a0 + 2 * lane
            UpRaw u;
            u.cm = seg[-1]; u.c01 = *reinterpret_cast<const float2*>(seg); u.cp = seg[2];
            up_row_raw(u, hp[p]);
        }
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            FineRaw<L0> rf;
            if (L0) {
                const CtStage<true>& T = reinterpret_cast<const CtStage<true>&>(S);
                fine_from_rows(reinterpret_cast<const float4*>(T.fine[0][r])[lane], reinterpret_cast<const float4*>(T.fine[1][r])[lane],
                               reinterpret_cast<const float4*>(T.mask[r])[lane], rf);
            } else {
                const CtStage<false>& T = reinterpret_cast<const CtStage<false>&>(S);
                fine_from_rows(reinterpret_cast<const float4*>(T.fine[c][r])[lane], reinterpret_cast<const float4*>(T.fine[3 + c][r])[lane],
                               reinterpret_cast<const float4*>(T.fine[6][r])[lane], rf);
            }
            fine_unpack(rf, c, gl[r], gr[r], mk[r]);
        }
        // the stage is in registers: release it to the producer
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->empty[s]);
        float e[4], o[4];
#pragma unroll
        for (int i = 0; i < 4; i += 2) {
            float2 u[3];
#pragma unroll
            for (int p = 0; p < 3; ++p)
                u[p] = up_even2(make_float2(hm[p][i], hm[p][i + 1]), make_float2(h0[p][i], h0[p][i + 1]),
                                make_float2(hp[p][i], hp[p][i + 1]), nz);
            const float2 ev = blend2(make_float2(gl[0][i], gl[0][i + 1]), make_float2(gr[0][i], gr[0][i + 1]),
                                     make_float2(mk[0][i], mk[0][i + 1]), u[0], u[1], u[2], nz);
            e[i] = ev.x; e[i + 1] = ev.y;
#pragma unroll
            for (int p = 0; p < 3; ++p)
                u[p] = up_odd2(make_float2(h0[p][i], h0[p][i + 1]), make_float2(hp[p][i], hp[p][i + 1]));
            const float2 ov = blend2(make_float2(gl[1][i], gl[1][i + 1]), make_float2(gr[1][i], gr[1][i + 1]),
                                     make_float2(mk[1][i], mk[1][i + 1]), u[0], u[1], u[2], nz);
            o[i] = ov.x; o[i + 1] = ov.y;
        }
        if (EMIT) {
            if (emit_words) emit_rows_interior(*E, k, e, o, c, lane, A.w, fy, fx0);
            else emit_rows_generic(*E, k, e, o, true, c, A.w, fy, fx);
        } else {
            *reinterpret_cast<float4*>(orow) = make_float4(e[0], e[1], e[2], e[3]);
            *reinterpret_cast<float4*>(orow + A.opitch) = make_float4(o[0], o[1], o[2], o[3]);
            orow += 2 * (size_t)A.opitch;
        }
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
            for (int i = 0; i < 4; ++i) { hm[p][i] = h0[p][i]; h0[p][i] = hp[p][i]; }
    }
}

// block (32, 4): warps 0-2 = colour channels, warp 3 = TMA producer; grid (ceil(w/128), ceil(h/32), frames).
// tm_fine: L0 -> the warped word planes [2 * frames][h][wpitch], else the fine Gaussian planes [7 * frames][h][fpitch];
// tm_mask (L0): the level-0 mask planes [frames][h][mpitch]; tm_gc / tm_oc: the coarse Gaussian / out planes.
template <bool L0, bool EMIT>
__global__ void __launch_bounds__(128, L0 ? 6 : 5)
k_collapse_tma(const __grid_constant__ TmaMap tm_fine, const __grid_constant__ TmaMap tm_mask, const __grid_constant__ TmaMap tm_gc,
               const __grid_constant__ TmaMap tm_oc, const uint32_t* __restrict__ warped, int wpitch, size_t wstride,
               const float* __restrict__ mask0, int mpitch, size_t m0stride, const float* __restrict__ g_fine, int w, int h, int fpitch,
               size_t fstride, const float* __restrict__ g_coarse, const float* __restrict__ out_coarse, int cw, int ch, int cpitch,
               size_t cstride, float* __restrict__ out_fine, int opitch, size_t ostride, const unsigned char* __restrict__ tile_flags,
               const FrameParams* __restrict__ fp, uint8_t* __restrict__ frames_base, size_t frame_bytes, unsigned char* __restrict__ ex,
               int ex_pitch, size_t ex_stride, int map_frame0, int R) {
    extern __shared__ __align__(128) unsigned char smem_dyn[];
    const int f = blockIdx.z, warp = threadIdx.y, lane = threadIdx.x, c = warp < 3 ? warp : 0;
    if (tile_flags && !tile_flags[((size_t)f * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x]) return;
    const int fx = blockIdx.x * 128 + 4 * lane, cy0 = blockIdx.y * R;
    CollapseArgs A;
    A.w1 = L0 ? warped + (size_t)f * 2 * wstride : nullptr; A.w2 = L0 ? A.w1 + wstride : nullptr; A.wpitch = wpitch;
    A.mask0 = L0 ? mask0 + (size_t)f * m0stride : nullptr; A.mpitch = mpitch;
    A.gfine = L0 ? nullptr : g_fine + (size_t)f * 7 * fstride; A.fpitch = fpitch; A.fstride = fstride;
    A.gc = g_coarse + (size_t)f * 7 * cstride; A.oc = out_coarse + (size_t)f * 3 * cstride;
    A.cw = cw; A.ch = ch; A.cpitch = cpitch; A.cstride = cstride;
    A.out = EMIT ? nullptr : out_fine + (size_t)f * 3 * ostride; A.opitch = opitch; A.ostride = ostride; A.w = w; A.h = h;
    CtStage<L0>* stages = reinterpret_cast<CtStage<L0>*>(smem_dyn);
    CtBars* bars = reinterpret_cast<CtBars*>(smem_dyn + CT_NS * sizeof(CtStage<L0>));
    EmitCtx E;
    bool emit_words = false;
    if (EMIT) {
        E.frame = frames_base + (size_t)fp[f].dst_slot * frame_bytes;
        E.ex = ex + ((size_t)f * 3 + c) * ex_stride; E.ex_pitch = ex_pitch;
        E.rowbuf = smem_dyn + CT_NS * sizeof(CtStage<L0>) + 128;
        E.excess = 0.f;
        emit_words = (w & 3) == 0 && (reinterpret_cast<size_t>(E.frame) & 3) == 0;
    }
    const int a = fx >> 1;
    const bool lane_in = a >= 1 && a + 2 <= cw - 1;                       // implies fx + 3 < w
    const bool rows_in = cy0 >= 1 && cy0 + R <= ch - 1 && 2 * (cy0 + R) <= h;
    if (__all_sync(FULL, lane_in && rows_in)) {                           // the same decision in all four warps
        if (warp == 3 && lane == 0) {
#pragma unroll
            for (int i = 0; i < CT_NS; ++i) { mbar_init(&bars->full[i], 1); mbar_init(&bars->empty[i], 3); }
            asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        }
        __syncthreads();
        if (warp == 3) {
            if (lane == 0) {
                const int fx0 = blockIdx.x * 128, a0 = fx0 >> 1, mf = map_frame0 + f;      // the maps span the whole chunk
#pragma unroll 1
                for (int k = 0; k < R; ++k) {
                    const int s = k % CT_NS;
                    if (k >= CT_NS) mbar_wait(&bars->empty[s], (unsigned)(k / CT_NS - 1) & 1u);
                    // the channel warps read the stage through the generic proxy; order those reads before the TMA writes
                    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
                    unsigned long long* bar = &bars->full[s];
                    mbar_expect_tx(bar, ct_stage_bytes<L0>());
                    CtStage<L0>& S = stages[s];
                    if (L0) {
                        CtStage<true>& T = reinterpret_cast<CtStage<true>&>(S);
                        tma_load_3d(T.fine, &tm_fine, fx0, 2 * (cy0 + k), 2 * mf, bar);
                        tma_load_3d(T.mask, &tm_mask, fx0, 2 * (cy0 + k), mf, bar);
                    } else {
                        CtStage<false>& T = reinterpret_cast<CtStage<false>&>(S);
                        tma_load_3d(T.fine, &tm_fine, fx0, 2 * (cy0 + k), 7 * mf, bar);
                    }
                    tma_load_3d(S.gc, &tm_gc, a0 - 4, cy0 + k + 1, 7 * mf, bar);
                    tma_load_3d(S.oc, &tm_oc, a0 - 4, cy0 + k + 1, 3 * mf, bar);
                }
            }
            return;
        }
        collapse_consume<L0, EMIT>(A, c, fx, cy0, lane, stages, bars, &E, emit_words, R);
    } else if (warp < 3 && fx < w) {
        collapse_body<L0, EMIT>(A, c, fx, cy0, &E, R);
    }
}

// ---- the tail of the pyramid in one launch ----------------------------------------------------------------------------
// Settings::pyramid_levels defaults to 64 (reference src/settings.hpp:20): a 512 x 512 frame reaches 1 x 1 at level 9 and the
// reference keeps calling pyrDown / pyrUp on 1 x 1 images for 55 more levels (OCV pyramids.cpp:945-950 handles them). Launching
// two kernels per level makes a chained frame launch-latency bound (~130 launches). k_pyramid_tail runs every level from k0
// (the first one no larger than 32 x 32) to L and back inside one CTA per frame: the same generic bodies as the per-level
// kernels (bit-identical), block barriers between the levels, L2-coherent loads for what the CTA itself wrote.
__global__ void __launch_bounds__(256)
k_pyramid_tail(float* __restrict__ g_base, float* __restrict__ o_base, const TailLevel* __restrict__ lv, int k0, int L) {
    const int f = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Gaussian pyramids (7 planes) down to level L
    for (int k = k0; k < L; ++k) {
        const TailLevel S = lv[k], D = lv[k + 1];
        const float* sb = g_base + S.g_off + (size_t)f * 7 * S.plane_stride;
        float* db = g_base + D.g_off + (size_t)f * 7 * D.plane_stride;
        const DownSel sel(S.w, D.w);
        const int ncol = div_up(D.w, 64), nrow = div_up(D.h, 4), jobs = 7 * ncol * nrow;
        for (int job = warp; job < jobs; job += 8) {
            const int p = job % 7, rest = job / 7, xo = 64 * (rest % ncol) + 2 * lane, y0 = 4 * (rest / ncol);
            const unsigned flags = down_pair_flags(sel, xo, p < 6, p % 3);
            if (xo < D.w)
                down_chunk_f32<false, 4, true>(sb + (size_t)p * S.plane_stride, S.w, S.h, S.pitch, db + (size_t)p * D.plane_stride, D.w, D.h,
                                               D.pitch, xo, y0, lane, flags);
        }
        // while a level is one job per plane, plane p stays with warp p from level to level: no block barrier needed
        if (jobs == 7 && k + 1 < L) __syncwarp(); else __syncthreads();
    }
    __syncthreads();
    {   // resultSmallest (blend.hpp:68-69)
        const TailLevel T = lv[L];
        const float* gf = g_base + T.g_off + (size_t)f * 7 * T.plane_stride;
        float* of = o_base + T.o_off + (size_t)f * 3 * T.plane_stride;
        for (int i = threadIdx.x; i < T.w * T.h; i += 256) {
            const size_t o = (size_t)(i / T.w) * T.pitch + (i % T.w);
            const float m = __ldca(gf + 6 * T.plane_stride + o), anti = __fsub_rn(1.0f, m);
#pragma unroll
            for (int c = 0; c < 3; ++c)
                of[(size_t)c * T.plane_stride + o] = __fadd_rn(__fmul_rn(__ldca(gf + (size_t)c * T.plane_stride + o), m),
                                                               __fmul_rn(__ldca(gf + (size_t)(3 + c) * T.plane_stride + o), anti));
        }
        __syncthreads();
    }
    // collapse back up to level k0
    for (int k = L - 1; k >= k0; --k) {
        const TailLevel F = lv[k], Cc = lv[k + 1];
        CollapseArgs A;
        A.w1 = A.w2 = nullptr; A.wpitch = 0; A.mask0 = nullptr; A.mpitch = 0;
        A.gfine = g_base + F.g_off + (size_t)f * 7 * F.plane_stride; A.fpitch = F.pitch; A.fstride = F.plane_stride;
        A.gc = g_base + Cc.g_off + (size_t)f * 7 * Cc.plane_stride; A.oc = o_base + Cc.o_off + (size_t)f * 3 * Cc.plane_stride;
        A.cw = Cc.w; A.ch = Cc.h; A.cpitch = Cc.pitch; A.cstride = Cc.plane_stride;
        A.out = o_base + F.o_off + (size_t)f * 3 * F.plane_stride; A.opitch = F.pitch; A.ostride = F.plane_stride; A.w = F.w; A.h = F.h;
        const int ncol = div_up(F.w, 128), nrow = div_up(F.h, 8), jobs = 3 * ncol * nrow;
        for (int job = warp; job < jobs; job += 8) {
            const int c = job % 3, rest = job / 3, fx = 128 * (rest % ncol) + 4 * lane, cy0 = 4 * (rest / ncol);
            if (fx < F.w) collapse_body<false, false, true>(A, c, fx, cy0, nullptr, 4);
        }
        // one job per channel: out[k] of channel c is written and read (as out_coarse of level k-1) by warp c; the Gaussian
        // planes were all finished before the barrier that precedes the collapse
        const int next_jobs = k > k0 ? 3 * div_up(lv[k - 1].w, 128) * div_up(lv[k - 1].h, 8) : 0;
        if (jobs == 3 && next_jobs == 3) __syncwarp(); else __syncthreads();
    }
}

void launch_pyr_down0(cudaStream_t st, const uint32_t* warped, int wpitch, size_t wstride, const float* basis, int bpitch,
                      const FrameParams* fp, int w, int h, float* mask0, size_t m0stride, float* dst, LevelDesc dl,
                      int frames) {
    const dim3 grid(div_up(dl.w, 128), div_up(dl.h, 3 * DN_R), 3 * frames), block(32, 3);
    static SmemAttrOnce done;
    ensure_smem_attr(k_pyr_down0_roll, D0_SMEM, done);
    k_pyr_down0_roll<<<grid, block, D0_SMEM, st>>>(warped, wpitch, wstride, basis, bpitch, fp, w, h, mask0, m0stride, dst, dl.w, dl.h,
                                                   dl.pitch, dl.plane_stride);
}

void launch_pyr_down0_seg(cudaStream_t st, const uint32_t* warped, int wpitch, size_t wstride, const SegFrame* seg, int bpitch,
                          const FrameParams* fp, int w, int h, float* mask0, size_t m0stride, float* dst, LevelDesc dl,
                          int frames) {
    const dim3 grid(div_up(dl.w, 128), div_up(dl.h, 3 * DN_R), 3 * frames), block(32, 3);
    static SmemAttrOnce done;
    ensure_smem_attr(k_pyr_down0_roll_seg, D0_SMEM, done);
    k_pyr_down0_roll_seg<<<grid, block, D0_SMEM, st>>>(warped, wpitch, wstride, seg, bpitch, fp, w, h, mask0, m0stride, dst, dl.w,
                                                       dl.h, dl.pitch, dl.plane_stride);
}

void launch_pyr_down(cudaStream_t st, const float* src, LevelDesc sl, float* dst, LevelDesc dl, int frames) {
    // a grid of 16-row walks that cannot give every SM a few CTAs is cut into 4-row walks instead
    const long long ctas16 = (long long)div_up(dl.w, 128) * div_up(dl.h, 4 * DN_R) * frames * 7;
    if (ctas16 < 148 * 12)
        k_pyr_down_roll<4><<<dim3(div_up(dl.w, 128), div_up(dl.h, 4 * 4), frames * 7), dim3(32, 4), 0, st>>>(
            src, sl.w, sl.h, sl.pitch, sl.plane_stride, dst, dl.w, dl.h, dl.pitch, dl.plane_stride);
    else
        k_pyr_down_roll<DN_R><<<dim3(div_up(dl.w, 128), div_up(dl.h, 4 * DN_R), frames * 7), dim3(32, 4), 0, st>>>(
            src, sl.w, sl.h, sl.pitch, sl.plane_stride, dst, dl.w, dl.h, dl.pitch, dl.plane_stride);
}

void launch_pyramid_tail(cudaStream_t st, float* g_base, float* o_base, const TailLevel* levels, int k0, int L, int frames) {
    k_pyramid_tail<<<frames, 256, 0, st>>>(g_base, o_base, levels, k0, L);
}

void launch_blend_coarsest(cudaStream_t st, const float* g, LevelDesc l, float* out, int frames) {
    k_blend_coarsest<<<dim3(div_up(l.w * l.h, 256), frames), 256, 0, st>>>(g, l.w, l.h, l.pitch, l.plane_stride, out);
}

void launch_collapse(cudaStream_t st, const float* g_fine, LevelDesc fl, const float* g_coarse, const float* out_coarse,
                     LevelDesc cl, float* out_fine, int frames, const CollapseMaps* maps) {
    // coarse rows per warp: 16 on the large levels; a grid of 16-row walks that cannot give every SM a few CTAs is cut into
    // 4-row walks (the small levels are pure latency: four times the warps, each a quarter as long)
    const long long ctas16 = (long long)div_up(fl.w, 128) * div_up(fl.h, 2 * CL_R) * frames;
    const int R = ctas16 < 148 * 12 ? 4 : CL_R;
    const dim3 grid(div_up(fl.w, 128), div_up(fl.h, 2 * R), frames);
    if (maps) {
        static SmemAttrOnce done;
        ensure_smem_attr(k_collapse_tma<false, false>, ct_smem<false, false>(), done);
        k_collapse_tma<false, false><<<grid, dim3(32, 4), ct_smem<false, false>(), st>>>(
            maps->fine, maps->mask, maps->gc, maps->oc, nullptr, 0, 0, nullptr, 0, 0, g_fine, fl.w, fl.h, fl.pitch, fl.plane_stride, g_coarse,
            out_coarse, cl.w, cl.h, cl.pitch, cl.plane_stride, out_fine, fl.pitch, fl.plane_stride, nullptr, nullptr, nullptr, 0, nullptr, 0, 0, 0,
            R);
        return;
    }
    k_collapse_roll<false, false><<<grid, dim3(32, 3), 0, st>>>(
        nullptr, 0, 0, nullptr, 0, 0, g_fine, fl.w, fl.h, fl.pitch, fl.plane_stride, g_coarse, out_coarse, cl.w, cl.h, cl.pitch,
        cl.plane_stride, out_fine, fl.pitch, fl.plane_stride, nullptr, nullptr, nullptr, 0, nullptr, 0, 0, R);
}

void launch_collapse0(cudaStream_t st, const uint32_t* warped, int wpitch, size_t wstride, const float* mask0, int mpitch,
                      size_t m0stride, int w, int h, const float* g_coarse, const float* out_coarse, LevelDesc cl,
                      float* out_fine, LevelDesc ol, int frames, const unsigned char* tile_flags, const CollapseMaps* maps) {
    const dim3 grid(div_up(w, 128), div_up(h, 2 * CL_R), frames);
    if (maps) {
        static SmemAttrOnce done;
        ensure_smem_attr(k_collapse_tma<true, false>, ct_smem<true, false>(), done);
        k_collapse_tma<true, false><<<grid, dim3(32, 4), ct_smem<true, false>(), st>>>(
            maps->fine, maps->mask, maps->gc, maps->oc, warped, wpitch, wstride, mask0, mpitch, m0stride, nullptr, w, h, 0, 0, g_coarse,
            out_coarse, cl.w, cl.h, cl.pitch, cl.plane_stride, out_fine, ol.pitch, ol.plane_stride, tile_flags, nullptr, nullptr, 0, nullptr,
            0, 0, 0, CL_R);
        return;
    }
    k_collapse_roll<true, false><<<grid, dim3(32, 3), 0, st>>>(
        warped, wpitch, wstride, mask0, mpitch, m0stride, nullptr, w, h, 0, 0, g_coarse, out_coarse, cl.w, cl.h, cl.pitch,
        cl.plane_stride, out_fine, ol.pitch, ol.plane_stride, tile_flags, nullptr, nullptr, 0, nullptr, 0, 0, CL_R);
}

void launch_collapse0_emit(cudaStream_t st, const uint32_t* warped, int wpitch, size_t wstride, const float* mask0, int mpitch,
                           size_t m0stride, int w, int h, const float* g_coarse, const float* out_coarse, LevelDesc cl,
                           const FrameParams* fp, uint8_t* frames_base, size_t frame_bytes, unsigned char* ex, int ex_pitch,
                           size_t ex_stride, int frames, const CollapseMaps* maps) {
    const dim3 grid(div_up(w, 128), div_up(h, 2 * CL_R), frames);
    if (maps) {
        static SmemAttrOnce done;
        ensure_smem_attr(k_collapse_tma<true, true>, ct_smem<true, true>(), done);
        k_collapse_tma<true, true><<<grid, dim3(32, 4), ct_smem<true, true>(), st>>>(
            maps->fine, maps->mask, maps->gc, maps->oc, warped, wpitch, wstride, mask0, mpitch, m0stride, nullptr, w, h, 0, 0, g_coarse,
            out_coarse, cl.w, cl.h, cl.pitch, cl.plane_stride, nullptr, 0, 0, nullptr, fp, frames_base, frame_bytes, ex, ex_pitch, ex_stride, 0,
            CL_R);
        return;
    }
    k_collapse_roll<true, true><<<grid, dim3(32, 3), 0, st>>>(
        warped, wpitch, wstride, mask0, mpitch, m0stride, nullptr, w, h, 0, 0, g_coarse, out_coarse, cl.w, cl.h, cl.pitch,
        cl.plane_stride, nullptr, 0, 0, nullptr, fp, frames_base, frame_bytes, ex, ex_pitch, ex_stride, CL_R);
}

}  // namespace poppy
