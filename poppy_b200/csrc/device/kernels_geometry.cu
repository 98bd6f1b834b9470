// Kernel group 1 — vertex lerp, per-triangle affine solve, and the exact triangle-ID rasteriser.
//
//   k_clip_points      clip_points()                        reference src/util.cpp:453-460
//   k_lerp_points      morph_points() + clip_points()       reference src/algo.cpp:50-58,202-205
//   k_tri_geometry     make_triangler_points, solve_homography, morph_homography, the Mat::inv of create_map
//                                                           reference src/algo.cpp:83-93,108-144,154-157
//                      + closed form of cv::FillConvexPoly's edge walkers (OCV drawing.cpp:1093-1255)
//   k_bin_scan/_fill   per-frame lists of the triangles touching each 64x32 screen tile (feeds k_raster_warp,
//                      kernels_warp.cu, which paints the triangle-ID tile in shared memory)
#include "common.cuh"
#include "kernels.cuh"

namespace poppy {

// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 clip_point(float2 p, int cols, int rows) {
    p.x = p.x > (float)cols ? (float)(cols - 1) : p.x;
    p.y = p.y > (float)rows ? (float)(rows - 1) : p.y;
    p.x = p.x < 0.f ? 0.f : p.x;
    p.y = p.y < 0.f ? 0.f : p.y;
    return p;
}

__global__ void k_clip_points(const float2* __restrict__ in, float2* __restrict__ out, int n, int cols, int rows) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = clip_point(in[i], cols, rows);
}

// x = (float)((1.0 - (double)s) * (double)a + (double)(float)(s * b))      (SURVEY.md A.8)
__device__ __forceinline__ float lerp_coord(float a, float b, float s) {
    float sb = __fmul_rn(s, b);
    double t = __dadd_rn(__dmul_rn(__dsub_rn(1.0, (double)s), (double)a), (double)sb);
    return __double2float_rn(t);
}

// grid (ceil(n/256), frames). Frame f reads p1 + f * p1_frame_stride (0: every frame starts from the same set)
// and writes out + f * out_frame_stride. SEG: frame f's pts2 and point count are its segment's (seg[f]); n is their maximum.
template <bool SEG>
__device__ __forceinline__ void lerp_points_body(const float2* __restrict__ p1, size_t p1_frame_stride, const float2* __restrict__ p2,
                                                 const FrameParams* __restrict__ fp, const SegFrame* __restrict__ seg,
                                                 float2* __restrict__ out, size_t out_frame_stride, int n, int cols, int rows) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int f = blockIdx.y;
    if (SEG) {
        n = seg[f].n_points;
        p2 = seg[f].pts2;
    }
    if (i >= n) return;
    float s = fp[f].shape;
    float2 a = p1[(size_t)f * p1_frame_stride + i], b = p2[i], r;
    r.x = lerp_coord(a.x, b.x, s);
    r.y = lerp_coord(a.y, b.y, s);
    out[(size_t)f * out_frame_stride + i] = clip_point(r, cols, rows);
}

__global__ void k_lerp_points(const float2* __restrict__ p1, size_t p1_frame_stride, const float2* __restrict__ p2,
                              const FrameParams* __restrict__ fp, float2* __restrict__ out, size_t out_frame_stride, int n,
                              int cols, int rows) {
    lerp_points_body<false>(p1, p1_frame_stride, p2, fp, nullptr, out, out_frame_stride, n, cols, rows);
}

__global__ void k_lerp_points_seg(const float2* __restrict__ p1, size_t p1_frame_stride, const SegFrame* __restrict__ seg,
                                  const FrameParams* __restrict__ fp, float2* __restrict__ out, size_t out_frame_stride, int n,
                                  int cols, int rows) {
    lerp_points_body<true>(p1, p1_frame_stride, nullptr, fp, seg, out, out_frame_stride, n, cols, rows);
}

// ------------------------------------------------------------------------------------------------------------------
// 3x3 float inverse via double cofactors, zero matrix when singular — OCV core/src/lapack.cpp:760-763,965-995,1045
__device__ void inv3(const float* m, float* o) {
#define M(r, c) ((double)m[(r) * 3 + (c)])
#define COF(a, b, c, d) __dsub_rn(__dmul_rn(a, b), __dmul_rn(c, d))
    double d = __dadd_rn(__dsub_rn(__dmul_rn(M(0, 0), COF(M(1, 1), M(2, 2), M(1, 2), M(2, 1))),
                                   __dmul_rn(M(0, 1), COF(M(1, 0), M(2, 2), M(1, 2), M(2, 0)))),
                         __dmul_rn(M(0, 2), COF(M(1, 0), M(2, 1), M(1, 1), M(2, 0))));
    if (d == 0.) {
#pragma unroll
        for (int i = 0; i < 9; ++i) o[i] = 0.f;
        return;
    }
    d = __ddiv_rn(1., d);
    o[0] = __double2float_rn(__dmul_rn(COF(M(1, 1), M(2, 2), M(1, 2), M(2, 1)), d));
    o[1] = __double2float_rn(__dmul_rn(COF(M(0, 2), M(2, 1), M(0, 1), M(2, 2)), d));
    o[2] = __double2float_rn(__dmul_rn(COF(M(0, 1), M(1, 2), M(0, 2), M(1, 1)), d));
    o[3] = __double2float_rn(__dmul_rn(COF(M(1, 2), M(2, 0), M(1, 0), M(2, 2)), d));
    o[4] = __double2float_rn(__dmul_rn(COF(M(0, 0), M(2, 2), M(0, 2), M(2, 0)), d));
    o[5] = __double2float_rn(__dmul_rn(COF(M(0, 2), M(1, 0), M(0, 0), M(1, 2)), d));
    o[6] = __double2float_rn(__dmul_rn(COF(M(1, 0), M(2, 1), M(1, 1), M(2, 0)), d));
    o[7] = __double2float_rn(__dmul_rn(COF(M(0, 1), M(2, 0), M(0, 0), M(2, 1)), d));
    o[8] = __double2float_rn(__dmul_rn(COF(M(0, 0), M(1, 1), M(0, 1), M(1, 0)), d));
#undef COF
#undef M
}

// 3x3 float product as the FMA-dispatched gemm evaluates it: fma(a2,b2, fma(a0,b0, a1*b1))
// (OCV core/src/matmul.simd.hpp:827-858, SURVEY.md A.5)
__device__ void mul3(const float* a, const float* b, float* o) {
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            float p1 = __fmul_rn(a[i * 3 + 1], b[3 + j]);
            o[i * 3 + j] = fmaf(a[i * 3 + 2], b[6 + j], fmaf(a[i * 3 + 0], b[j], p1));
        }
}

// Closed form of the scan-fill state machine of cv::FillConvexPoly for a triangle (drawing.cpp:1163-1252):
// which rows are span-filled and where the two edge walkers are on each of them.
__device__ void make_fill_record(TriRaster& r, int img_h) {
    const int n = 3;
    int imin = 0, ymin = r.vy[0], ymax = r.vy[0];
#pragma unroll
    for (int i = 1; i < n; ++i) {
        if (r.vy[i] < ymin) { ymin = r.vy[i]; imin = i; }
        ymax = max(ymax, r.vy[i]);
    }
    ymax = min(ymax, img_h - 1);
    int idx[2] = {imin, imin}, ye[2] = {ymin, ymin}, nseg[2] = {0, 0};
    const int di[2] = {1, n - 1};
    r.sw[0] = r.sw[1] = 32767;
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) { r.x0[i][j] = -65536; r.dx[i][j] = 0; }
    int y = ymin, edges = n, yend = ymax + 1;
    for (;;) {
        for (int i = 0; i < 2; ++i) {
            if (y < ye[i]) continue;
            int from = idx[i], to = from + di[i];
            if (to >= n) to -= n;
            while (edges-- > 0) {
                int ty = r.vy[to];
                if (ty > y) {
                    long long xs = (long long)r.vx[from] << 16, xe = (long long)r.vx[to] << 16;
                    int j = min(nseg[i], 1);
                    r.x0[i][j] = (int)xs;
                    r.dx[i][j] = (int)(((xe - xs) * 2 + (ty - y)) / (2 * (ty - y)));
                    if (j == 1) r.sw[i] = (short)y;
                    nseg[i]++;
                    ye[i] = ty;
                    idx[i] = to;
                    break;
                }
                from = to;
                to += di[i];
                if (to >= n) to -= n;
            }
        }
        if (edges < 0) { yend = y; break; }
        int ynext = min(ye[0], ye[1]);
        if (ynext > ymax) break;           // both walkers run to the last row
        y = ynext;
    }
    r.ymin = (short)ymin;
    r.yend = (short)yend;
}

// Screen tiles (RW_TW x RW_TH pixels) a triangle's bounding box touches; false when it lies outside the image.
__device__ __forceinline__ bool tile_bbox(const TriRaster& r, int w, int h, int& tx0, int& tx1, int& ty0, int& ty1) {
    const int x0 = max(min(min(r.vx[0], r.vx[1]), r.vx[2]), 0), x1 = min(max(max(r.vx[0], r.vx[1]), r.vx[2]), w - 1);
    const int y0 = max(min(min(r.vy[0], r.vy[1]), r.vy[2]), 0), y1 = min(max(max(r.vy[0], r.vy[1]), r.vy[2]), h - 1);
    if (x0 > x1 || y0 > y1) return false;
    tx0 = x0 / RW_TW; tx1 = x1 / RW_TW; ty0 = y0 / RW_TH; ty1 = y1 / RW_TH;
    return true;
}

// grid (ceil(max_tri/128), frames). tile_counts (frames x n_tiles, zeroed by the caller) receives, per screen tile,
// the number of triangles whose bounding box touches it. SEG: frame f's pts2 is its segment's (seg[f]).
template <bool SEG>
__device__ __forceinline__ void tri_geometry_body(const int3* __restrict__ tri_idx, const FrameParams* __restrict__ fp,
                                                  const float2* __restrict__ p1, size_t p1_frame_stride, const float2* __restrict__ p2,
                                                  const SegFrame* __restrict__ seg, const float2* __restrict__ morphed,
                                                  size_t morphed_frame_stride, int max_tri, int img_w, int img_h,
                                                  TriInverse* __restrict__ inv_out, TriRaster* __restrict__ rast_out,
                                                  int* __restrict__ tile_counts, int tiles_x, int n_tiles) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    int f = blockIdx.y;
    FrameParams P = fp[f];
    if (t >= P.n_tri) return;
    if (SEG) p2 = seg[f].pts2;
    int3 id = tri_idx[P.tri_base + t];
    const float2* s1 = p1 + (size_t)f * p1_frame_stride;
    const float2* mp = morphed + (size_t)f * morphed_frame_stride;
    int v[3] = {id.x, id.y, id.z};
    float P1[9], P2[9];
    TriRaster R;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float2 a = s1[v[k]], b = p2[v[k]], m = mp[v[k]];
        // cv::Point(float, float): truncation toward zero (reference src/algo.cpp:89)
        P1[k] = (float)__float2int_rz(a.x); P1[3 + k] = (float)__float2int_rz(a.y); P1[6 + k] = 1.f;
        P2[k] = (float)__float2int_rz(b.x); P2[3 + k] = (float)__float2int_rz(b.y); P2[6 + k] = 1.f;
        R.vx[k] = __float2int_rz(m.x); R.vy[k] = __float2int_rz(m.y);
    }
    make_fill_record(R, img_h);
    rast_out[(size_t)f * max_tri + t] = R;
    {
        int tx0, tx1, ty0, ty1;
        if (tile_bbox(R, img_w, img_h, tx0, tx1, ty0, ty1))
            for (int ty = ty0; ty <= ty1; ++ty)
                for (int tx = tx0; tx <= tx1; ++tx) atomicAdd(&tile_counts[(size_t)f * n_tiles + ty * tiles_x + tx], 1);
    }

    float iP1[9], H[9], iH[9], M1[9], M2[9];
    inv3(P1, iP1);
    mul3(P2, iP1, H);          // H = P2 * inv(P1)                       (algo.cpp:110)
    inv3(H, iH);
    const float r = P.shape, omr = P.one_minus_r;
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        float eye = (i % 4 == 0) ? 1.f : 0.f;
        M1[i] = fmaf(H[i], r, __fmul_rn(eye, omr));      // eye*(1-r) + H*r    via scaleAdd_32f (algo.cpp:130)
        M2[i] = fmaf(iH[i], omr, __fmul_rn(eye, r));     // eye*r + inv(H)*(1-r)               (algo.cpp:131)
    }
    TriInverse out;
    inv3(M1, out.a);
    inv3(M2, out.b);
    out.pad_a[0] = out.pad_a[1] = out.pad_a[2] = out.pad_b[0] = out.pad_b[1] = out.pad_b[2] = 0.f;
    inv_out[(size_t)f * max_tri + t] = out;
}

__global__ void k_tri_geometry(const int3* __restrict__ tri_idx, const FrameParams* __restrict__ fp,
                               const float2* __restrict__ p1, size_t p1_frame_stride, const float2* __restrict__ p2,
                               const float2* __restrict__ morphed, size_t morphed_frame_stride, int max_tri, int img_w,
                               int img_h, TriInverse* __restrict__ inv_out, TriRaster* __restrict__ rast_out,
                               int* __restrict__ tile_counts, int tiles_x, int n_tiles) {
    tri_geometry_body<false>(tri_idx, fp, p1, p1_frame_stride, p2, nullptr, morphed, morphed_frame_stride, max_tri, img_w, img_h,
                             inv_out, rast_out, tile_counts, tiles_x, n_tiles);
}

__global__ void k_tri_geometry_seg(const int3* __restrict__ tri_idx, const FrameParams* __restrict__ fp,
                                   const float2* __restrict__ p1, size_t p1_frame_stride, const SegFrame* __restrict__ seg,
                                   const float2* __restrict__ morphed, size_t morphed_frame_stride, int max_tri, int img_w,
                                   int img_h, TriInverse* __restrict__ inv_out, TriRaster* __restrict__ rast_out,
                                   int* __restrict__ tile_counts, int tiles_x, int n_tiles) {
    tri_geometry_body<true>(tri_idx, fp, p1, p1_frame_stride, nullptr, seg, morphed, morphed_frame_stride, max_tri, img_w, img_h,
                            inv_out, rast_out, tile_counts, tiles_x, n_tiles);
}

// ------------------------------------------------------------------------------------------------------------------
// Tile binning. k_bin_scan: per frame, exclusive prefix sum of the tile counts -> tile_off (n_tiles + 1 entries);
// a frame whose lists would not fit `cap` entries is flagged (the raster kernel then tests every triangle).
// block 1024; grid frames.
__global__ void __launch_bounds__(1024)
k_bin_scan(const int* __restrict__ tile_counts, int n_tiles, int cap, int* __restrict__ tile_off, int* __restrict__ overflow) {
    __shared__ int warp_sums[32];
    __shared__ int carry_s;
    const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int* cnt = tile_counts + (size_t)f * n_tiles;
    int* off = tile_off + (size_t)f * (n_tiles + 1);
    if (tid == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < n_tiles; base += 1024) {
        const int i = base + tid;
        const int v = i < n_tiles ? cnt[i] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        if (lane == 31) warp_sums[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int ws = warp_sums[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int n = __shfl_up_sync(0xffffffffu, ws, o);
                if (lane >= o) ws += n;
            }
            warp_sums[lane] = ws;
        }
        __syncthreads();
        const int carry = carry_s;
        const int excl = carry + (warp ? warp_sums[warp - 1] : 0) + incl - v;
        if (i < n_tiles) off[i] = excl;
        __syncthreads();
        if (tid == 1023) carry_s = carry + warp_sums[31];
        __syncthreads();
    }
    if (tid == 0) {
        off[n_tiles] = carry_s;
        overflow[f] = carry_s > cap ? 1 : 0;
    }
}

// grid (ceil(max_tri/128), frames): scatter triangle ids into their tiles' lists; tile_counts is consumed as the
// fill cursor (counted down to zero).
__global__ void k_bin_fill(const TriRaster* __restrict__ rast, const FrameParams* __restrict__ fp, int max_tri, int img_w,
                           int img_h, int* __restrict__ tile_counts, const int* __restrict__ tile_off,
                           const int* __restrict__ overflow, int* __restrict__ tile_list, int cap, int tiles_x, int n_tiles) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x, f = blockIdx.y;
    if (t >= fp[f].n_tri || overflow[f]) return;
    const TriRaster& R = rast[(size_t)f * max_tri + t];
    TriRaster r;
#pragma unroll
    for (int k = 0; k < 3; ++k) { r.vx[k] = R.vx[k]; r.vy[k] = R.vy[k]; }
    int tx0, tx1, ty0, ty1;
    if (!tile_bbox(r, img_w, img_h, tx0, tx1, ty0, ty1)) return;
    for (int ty = ty0; ty <= ty1; ++ty)
        for (int tx = tx0; tx <= tx1; ++tx) {
            const int tile = ty * tiles_x + tx;
            const int pos = atomicSub(&tile_counts[(size_t)f * n_tiles + tile], 1) - 1;
            tile_list[(size_t)f * cap + tile_off[(size_t)f * (n_tiles + 1) + tile] + pos] = t;
        }
}

// ------------------------------------------------------------------------------------------------------------------
void launch_clip_points(cudaStream_t st, const float2* in, float2* out, int n, int cols, int rows) {
    if (n > 0) k_clip_points<<<div_up(n, 256), 256, 0, st>>>(in, out, n, cols, rows);
}

void launch_lerp_points(cudaStream_t st, const float2* p1, size_t p1_frame_stride, const float2* p2,
                        const FrameParams* fp, float2* out, size_t out_frame_stride, int n, int frames, int cols,
                        int rows) {
    if (n > 0)
        k_lerp_points<<<dim3(div_up(n, 256), frames), 256, 0, st>>>(p1, p1_frame_stride, p2, fp, out, out_frame_stride,
                                                                    n, cols, rows);
}

void launch_tri_geometry(cudaStream_t st, const int3* tri_idx, const FrameParams* fp, const float2* p1,
                         size_t p1_frame_stride, const float2* p2, const float2* morphed, size_t morphed_frame_stride,
                         int max_tri, int tri_in_chunk_max, int frames, int img_w, int img_h, TriInverse* inv_out,
                         TriRaster* rast_out, int* tile_counts) {
    const int tiles_x = div_up(img_w, RW_TW), n_tiles = tiles_x * div_up(img_h, RW_TH);
    if (tri_in_chunk_max > 0)
        k_tri_geometry<<<dim3(div_up(tri_in_chunk_max, 128), frames), 128, 0, st>>>(
            tri_idx, fp, p1, p1_frame_stride, p2, morphed, morphed_frame_stride, max_tri, img_w, img_h, inv_out, rast_out,
            tile_counts, tiles_x, n_tiles);
}

void launch_lerp_points_seg(cudaStream_t st, const float2* p1, size_t p1_frame_stride, const SegFrame* seg,
                            const FrameParams* fp, float2* out, size_t out_frame_stride, int n_max, int frames, int cols,
                            int rows) {
    if (n_max > 0)
        k_lerp_points_seg<<<dim3(div_up(n_max, 256), frames), 256, 0, st>>>(p1, p1_frame_stride, seg, fp, out, out_frame_stride,
                                                                            n_max, cols, rows);
}

void launch_tri_geometry_seg(cudaStream_t st, const int3* tri_idx, const FrameParams* fp, const float2* p1,
                             size_t p1_frame_stride, const SegFrame* seg, const float2* morphed, size_t morphed_frame_stride,
                             int max_tri, int tri_in_chunk_max, int frames, int img_w, int img_h, TriInverse* inv_out,
                             TriRaster* rast_out, int* tile_counts) {
    const int tiles_x = div_up(img_w, RW_TW), n_tiles = tiles_x * div_up(img_h, RW_TH);
    if (tri_in_chunk_max > 0)
        k_tri_geometry_seg<<<dim3(div_up(tri_in_chunk_max, 128), frames), 128, 0, st>>>(
            tri_idx, fp, p1, p1_frame_stride, seg, morphed, morphed_frame_stride, max_tri, img_w, img_h, inv_out, rast_out,
            tile_counts, tiles_x, n_tiles);
}

void launch_bin_triangles(cudaStream_t st, const TriRaster* rast, const FrameParams* fp, int max_tri, int tri_in_chunk_max,
                          int frames, int img_w, int img_h, int* tile_counts, int* tile_off, int* overflow, int* tile_list,
                          int cap) {
    const int tiles_x = div_up(img_w, RW_TW), n_tiles = tiles_x * div_up(img_h, RW_TH);
    k_bin_scan<<<frames, 1024, 0, st>>>(tile_counts, n_tiles, cap, tile_off, overflow);
    if (tri_in_chunk_max > 0)
        k_bin_fill<<<dim3(div_up(tri_in_chunk_max, 128), frames), 128, 0, st>>>(rast, fp, max_tri, img_w, img_h, tile_counts,
                                                                              tile_off, overflow, tile_list, cap, tiles_x,
                                                                              n_tiles);
}

}  // namespace poppy
