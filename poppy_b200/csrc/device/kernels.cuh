// Host-callable launchers of the device kernels (one per kernel class). All launches go to the given stream.
#pragma once

#include <atomic>

#include "common.cuh"

namespace poppy {

// Opt-in to > 48 KB of dynamic shared memory, once per device and kernel: cudaFuncSetAttribute applies to the current
// device only, and one process may hold contexts on several GPUs (poppy_cuda.h: one context per GPU, thread-safe).
struct SmemAttrOnce { std::atomic<bool> done[64]; };
template <class K>
inline void ensure_smem_attr(K kernel, size_t bytes, SmemAttrOnce& once) {
    int dev = 0;
    cudaGetDevice(&dev);
    const bool tracked = dev >= 0 && dev < 64;
    if (!tracked || !once.done[dev].load(std::memory_order_acquire)) {
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (tracked) once.done[dev].store(true, std::memory_order_release);
    }
}

// A CUtensorMap (cuda.h), kept opaque here: built on the host by cuTensorMapEncodeTiled (poppy_cuda.cu), passed to the
// kernels as a __grid_constant__ parameter and named by cp.async.bulk.tensor.
struct alignas(64) TmaMap { unsigned long long v[16]; };
// The four box sources of one level's collapse (k_collapse_tma): fine level (warped word planes at level 0, the Gaussian
// planes otherwise), level-0 mask (level 0 only), coarse Gaussian planes, coarse out planes.
struct CollapseMaps { TmaMap fine, mask, gc, oc; };

// ---- kernels_geometry.cu -----------------------------------------------------------------------------------------
void launch_clip_points(cudaStream_t st, const float2* in, float2* out, int n, int cols, int rows);
void launch_lerp_points(cudaStream_t st, const float2* p1, size_t p1_frame_stride, const float2* p2,
                        const FrameParams* fp, float2* out, size_t out_frame_stride, int n, int frames, int cols,
                        int rows);
void launch_tri_geometry(cudaStream_t st, const int3* tri_idx, const FrameParams* fp, const float2* p1,
                         size_t p1_frame_stride, const float2* p2, const float2* morphed, size_t morphed_frame_stride,
                         int max_tri, int tri_in_chunk_max, int frames, int img_w, int img_h, TriInverse* inv_out,
                         TriRaster* rast_out, int* tile_counts);
// Segment renders: frame f of the chunk takes pts2 and its point count from seg[f] (n_max: the largest count of the chunk)
void launch_lerp_points_seg(cudaStream_t st, const float2* p1, size_t p1_frame_stride, const SegFrame* seg,
                            const FrameParams* fp, float2* out, size_t out_frame_stride, int n_max, int frames, int cols,
                            int rows);
void launch_tri_geometry_seg(cudaStream_t st, const int3* tri_idx, const FrameParams* fp, const float2* p1,
                             size_t p1_frame_stride, const SegFrame* seg, const float2* morphed, size_t morphed_frame_stride,
                             int max_tri, int tri_in_chunk_max, int frames, int img_w, int img_h, TriInverse* inv_out,
                             TriRaster* rast_out, int* tile_counts);
// tile_counts (frames x n_tiles, filled by launch_tri_geometry) -> tile_off (frames x (n_tiles+1)), overflow (frames),
// tile_list (frames x cap)
void launch_bin_triangles(cudaStream_t st, const TriRaster* rast, const FrameParams* fp, int max_tri, int tri_in_chunk_max,
                          int frames, int img_w, int img_h, int* tile_counts, int* tile_off, int* overflow, int* tile_list,
                          int cap);

// ---- kernels_warp.cu ---------------------------------------------------------------------------------------------
// BGR (3 bytes/px, tight rows) -> BGRX uchar4
void launch_bgr_to_bgrx(cudaStream_t st, const uint8_t* bgr, uchar4* out, int w, int h);
// every frame of a chunk: ring slot fp[f].dst_slot (BGR) -> out + f * w * h (BGRX)
void launch_bgr_to_bgrx_frames(cudaStream_t st, const uint8_t* frames_base, size_t frame_bytes, const FrameParams* fp, uchar4* out,
                               int w, int h, int frames);
// mask basis m2 = 1 - gray(gabor2)  (reference src/algo.cpp:250-252), rows `bpitch` floats apart
void launch_mask_basis(cudaStream_t st, const float* gabor_bgr, float* m2, int bpitch, int w, int h);

// ---- margin.cu ---------------------------------------------------------------------------------------------------
// the same basis derived from the 8-bit corrected2 (BGR, tight rows) as the reference derives gabor2 from it:
// 1 - gray(gabor_filter(corrected2 * 1/255)) with the default Gabor parameters (reference src/poppy.hpp:119-122); the first
// call on a device uploads the filter taps and synchronises `st`
cudaError_t launch_gabor_mask_basis(cudaStream_t st, const uint8_t* bgr, float* m2, int bpitch, int w, int h);
// paint_triangles + create_map + remap for both images, one CTA per 64x32 screen tile (reference src/algo.cpp:95-106,
// 146-176, 232-238). warped: per frame two planes of packed BGRX words (remap of image 1, of image 2), rows `wpitch`
// words apart, `wstride` words per plane; tri_map_out (nullable) receives frame 0's ID map. src1/src2: point-sampled,
// border-addressed (zero) uchar4 BGRX textures over cudaArrayTextureGather arrays, unnormalised coordinates
void launch_raster_warp(cudaStream_t st, const TriRaster* rast, const TriInverse* inv, const FrameParams* fp, int max_tri,
                        const int* tile_off, const int* tile_list, int cap, const int* overflow,
                        cudaTextureObject_t src1, cudaTextureObject_t src2, uint32_t* warped, int wpitch, size_t wstride, int* tri_map_out, int w, int h,
                        int frames);
// the same with frame f sampling its segment's textures seg[f].src1 / seg[f].src2 (no ID-map dump)
void launch_raster_warp_seg(cudaStream_t st, const TriRaster* rast, const TriInverse* inv, const FrameParams* fp, int max_tri,
                            const int* tile_off, const int* tile_list, int cap, const int* overflow, const SegFrame* seg,
                            uint32_t* warped, int wpitch, size_t wstride, int w, int h, int frames);

// ---- kernels_pyramid.cu ------------------------------------------------------------------------------------------
// level 0 -> 1: sources are the warped 8-bit pair (converted on the fly, algo.cpp:247-248) and the frame's blend
// mask evaluated from the mask basis (algo.cpp:255-258); the level-0 mask is also kept in mask0 (per-frame planes,
// rows bpitch floats apart, m0stride floats per frame) for launch_collapse0
void launch_pyr_down0(cudaStream_t st, const uint32_t* warped, int wpitch, size_t wstride, const float* basis, int bpitch,
                      const FrameParams* fp, int w, int h, float* mask0, size_t m0stride, float* dst, LevelDesc dl,
                      int frames);
// the same with frame f's mask basis seg[f].basis (rows bpitch floats apart)
void launch_pyr_down0_seg(cudaStream_t st, const uint32_t* warped, int wpitch, size_t wstride, const SegFrame* seg, int bpitch,
                          const FrameParams* fp, int w, int h, float* mask0, size_t m0stride, float* dst, LevelDesc dl,
                          int frames);
// level k -> k+1 for the 7 planes (left BGR, right BGR, mask)
void launch_pyr_down(cudaStream_t st, const float* src, LevelDesc sl, float* dst, LevelDesc dl, int frames);
// Levels k0 .. L of a chunk in one launch (one CTA per frame): pyrDown k0 -> ... -> L, resultSmallest, collapse L-1 .. k0.
// levels[k]: geometry of level k and the float offsets of its first plane inside the chunk's Gaussian / out blocks.
struct TailLevel { int w, h, pitch, pad; size_t plane_stride, g_off, o_off; };
void launch_pyramid_tail(cudaStream_t st, float* g_base, float* o_base, const TailLevel* levels, int k0, int L, int frames);
// resultSmallest = left*mask + right*(1-mask) at the coarsest level (blend.hpp:68-69)
void launch_blend_coarsest(cudaStream_t st, const float* g, LevelDesc l, float* out, int frames);
// out[k] = pyrUp(out[k+1]) + (G_l[k]-pyrUp(G_l[k+1]))*m[k] + (G_r[k]-pyrUp(G_r[k+1]))*(1-m[k])   (blend.hpp:45-77)
// maps (nullable): tensor maps of the level's planes; with them interior tiles are fed by a TMA producer warp, without them
// (levels too small to have an interior tile) every tile runs the generic body
void launch_collapse(cudaStream_t st, const float* g_fine, LevelDesc fl, const float* g_coarse, const float* out_coarse,
                     LevelDesc cl, float* out_fine, int frames, const CollapseMaps* maps);
// same for level 0, whose Gaussian level is the warped 8-bit pair + the level-0 mask planes
// tile_flags (nullable): per frame and 128x32 tile, 0 = the tile is not needed (calm, see below)
void launch_collapse0(cudaStream_t st, const uint32_t* warped, int wpitch, size_t wstride, const float* mask0, int mpitch,
                      size_t m0stride, int w, int h, const float* g_coarse, const float* out_coarse, LevelDesc cl,
                      float* out_fine, LevelDesc ol, int frames, const unsigned char* tile_flags, const CollapseMaps* maps);
// level-0 collapse fused with convertTo(CV_8U, 255): stores cvRound(255 out[0]) into the frame ring (exactly the frame
// wherever unsharp_mask() leaves the pixel untouched) and, per 4x8-pixel block and channel, whether out[0] left [0, 1] by
// more than 0.001 there: ex[(f*3 + c) * ex_stride + by * ex_pitch + bx]
void launch_collapse0_emit(cudaStream_t st, const uint32_t* warped, int wpitch, size_t wstride, const float* mask0, int mpitch,
                           size_t m0stride, int w, int h, const float* g_coarse, const float* out_coarse, LevelDesc cl,
                           const FrameParams* fp, uint8_t* frames_base, size_t frame_bytes, unsigned char* ex, int ex_pitch,
                           size_t ex_stride, int frames, const CollapseMaps* maps);

// ---- kernels_unsharp.cu ------------------------------------------------------------------------------------------
// unsharp_mask(lapBlend, 1, amount, 0.3) + convertTo(CV_8U, 255)   (reference src/algo.cpp:263-265, util.cpp:113-148)
// chunk_rows: rows per CTA (multiple of 8); chunk_flags (nullable): per frame and (strip, chunk), 0 = skip
void launch_unsharp_store(cudaStream_t st, const float* lap_blend, LevelDesc l, const FrameParams* fp,
                          uint8_t* frames_base, size_t frame_bytes, int frames, int chunk_rows,
                          const unsigned char* chunk_flags);
// Calm analysis between the fused level-0 collapse and the exact unsharp path (see EmitCtx, kernels_pyramid.cu): bounds
// |x - GaussianBlur(x)| from the second differences of the stored frame bytes and the clamp-excess flags. Outputs (per
// frame): block_dev [ceil(h/8)][ceil(w/4)][2] the per-block deviation maxima (scratch), block_flags [ceil(h/8)][ceil(w/4)] = 1
// where a 4x8 block fails the bound, chunk_flags
// [ceil(h/chunk_rows)][ceil(w/120)] = 1 where a strip chunk of launch_unsharp_store holds a pixel that unsharp_mask() may
// change, tile_flags [ceil(h/32)][ceil(w/128)] = 1 where a level-0 collapse tile is read by such a chunk; counts[f] =
// flagged chunks of frame f, *total += all of them (statistics). force_all: flag everything (exact path everywhere).
void launch_calm_analysis(cudaStream_t st, const uint8_t* frames_base, size_t frame_bytes, const FrameParams* fp,
                          const unsigned char* ex, int ex_pitch, size_t ex_stride, int w, int h, int frames, int chunk_rows,
                          unsigned char* block_dev, unsigned char* block_flags, unsigned char* chunk_flags,
                          unsigned char* tile_flags, int* counts, unsigned long long* total, int force_all);
constexpr int UNSHARP_STRIP_W = 120;       // output columns per strip of launch_unsharp_store
constexpr int CALM_BLOCK_W = 4, CALM_BLOCK_H = 8;
// order-dependent checksum of a byte range
void launch_checksum(cudaStream_t st, const uint8_t* data, size_t bytes, unsigned long long* out);

}  // namespace poppy
