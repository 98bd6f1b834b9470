// Shared device-side declarations of the sm_100a morph renderer.
//
// Numerics contract: every kernel reproduces the reference's CPU arithmetic bit for bit (SURVEY.md Appendix A).
// The whole device code is compiled with -fmad=false so that nvcc never contracts a*b+c on its own; an FMA is
// used exactly where the reference's FMA-dispatched OpenCV translation units fuse (fmaf()/fma() spelled out),
// and nowhere else.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace poppy {

// Per-frame scalars of one morph_images() call (reference src/algo.cpp:178): uploaded once per chunk.
struct FrameParams {
    float shape;        // (float)shapeRatio, the narrowing done by morph_points()/morph_homography()
    float one_minus_r;  // (float)(1.0 - (double)shape)
    double mask_alpha;  // 1.0 - maskRatio   (addWeighted alpha, algo.cpp:256)
    double mask_beta;   // -maskRatio        (addWeighted beta)
    float amount;       // (float)(1.0 - sin(maskRatio * pi)), algo.cpp:263-264
    int n_tri;          // triangles of this frame
    int tri_base;       // first triangle of this frame in the chunk's concatenated index list
    int dst_slot;       // frame ring slot written by the last stage
};

// Per-frame inputs of a segment render (poppy_cuda_render_segments): a chunk holds one step of several segments, and
// each frame reads its own segment's pair, mask basis and end points. Uploaded with the chunk's FrameParams.
struct __align__(8) SegFrame {
    cudaTextureObject_t src1;   // the segment's corrected1 at step 0, its chain array (the previous step's frame) after
    cudaTextureObject_t src2;   // the segment's corrected2
    const float* basis;         // the segment's mask basis, rows pitch0 floats apart
    const float2* pts2;         // the segment's clipped pts2
    int n_points;               // the segment's point count
    int pad;
};
static_assert(sizeof(SegFrame) == 40, "SegFrame layout");

// Raster record of one morphed triangle: integer vertices and the closed form of cv::FillConvexPoly's two edge
// walkers (OCV imgproc/src/drawing.cpp:1093-1255). 64 bytes.
struct __align__(16) TriRaster {
    int vx[3];          // truncated morphed vertices (reference src/algo.cpp:83-93)
    int vy[3];
    short ymin, yend;   // scan rows [ymin, yend) are span-filled (the row where the walkers run out is not)
    short sw[2];        // first row of walker i's second segment (32767 = none)
    int x0[2][2];       // 16.16 start x of walker i, segment j
    int dx[2][2];       // 16.16 per-row increment
};
static_assert(sizeof(TriRaster) == 64, "TriRaster layout");

// The two inverse matrices create_map() applies per pixel (reference src/algo.cpp:154-175). 96 bytes: each matrix is
// three aligned 16-byte loads for the warps that sample its image.
struct __align__(16) TriInverse {
    float a[9];         // inv(M1): maps a morphed-frame pixel into image 1
    float pad_a[3];
    float b[9];         // inv(M2): maps it into image 2
    float pad_b[3];
};
static_assert(sizeof(TriInverse) == 96, "TriInverse layout");

// One pyramid level of a frame chunk. Planes are row-major with `pitch` floats per row; plane p of frame f
// starts at base + ((size_t)f * planes + p) * plane_stride.
struct LevelDesc {
    int w, h, pitch;
    size_t plane_stride;   // pitch * h
};

__host__ __device__ inline int div_up(int a, int b) { return (a + b - 1) / b; }

// Screen tile of the fused rasterise-and-warp kernel (one CTA per tile) and of the triangle binning that feeds it.
constexpr int RW_TW = 64, RW_TH = 32;

// cv::borderInterpolate(BORDER_REFLECT_101), OCV core/src/copy.cpp:748-793
__device__ __forceinline__ int reflect101(int p, int len) {
    if ((unsigned)p < (unsigned)len) return p;
    if (len == 1) return 0;
    do {
        if (p < 0) p = -p;
        else p = 2 * len - 2 - p;
    } while ((unsigned)p >= (unsigned)len);
    return p;
}

// cvRound(float) as x86 cvtss2si evaluates it: round-half-even, INT_MIN when not representable
__device__ __forceinline__ int cv_round(float v) {
    return (fabsf(v) < 2147483648.0f) ? __float2int_rn(v) : (int)0x80000000;
}

}  // namespace poppy
