/* poppy_host.h — C ABI of the host stages that stay on the CPU (north-star): point hygiene, the Delaunay
 * topology of the morphed points, the vertex-index lookup and the frame schedule. Together with poppy_cuda.h this
 * is everything poppy::morph_images() does (reference src/algo.cpp:178-273); the C++ shim in
 * poppy_b200/csrc/host/morph_images.hpp keeps the reference's C++ signature on top of it.
 *
 * Replaced reference interfaces:
 *   clip_points / make_uniq / check_points          src/util.cpp:453-471,541-548
 *   morph_points                                    src/algo.cpp:50-58   (host copy; the device recomputes it bit-identically)
 *   cv::Subdiv2D::insert / getTriangleList          OCV imgproc/src/subdivision2d.cpp:412-490,756-785
 *   get_triangle_indices                            src/algo.cpp:60-81
 *   frame schedule of morph<Twriter>()              src/poppy.hpp:177-210
 */
#ifndef POPPY_HOST_H_
#define POPPY_HOST_H_

#include <stddef.h>
#include <stdint.h>

#include "poppy_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct poppy_host_plan poppy_host_plan;

/* clip both sets, lerp with (float)shape_ratio, clip the result: the morphedPoints of morph_images. */
int poppy_host_morph_points(const float* pts1_xy, const float* pts2_xy, int n, double shape_ratio, int width,
                            int height, float* out_xy);

/* clip -> make_uniq -> Delaunay -> triangle vertex indices into pts (first exact-equal occurrence), in
 * cv::Subdiv2D::getTriangleList order. *n_tri receives the triangle count even when it exceeds `cap`
 * (then POPPY_CUDA_ERR_CAPACITY is returned). POPPY_CUDA_ERR_INVALID where cv::Subdiv2D would throw
 * (a point with x >= width or y >= height after clipping). */
int poppy_host_triangulate(const float* pts_xy, int n, int width, int height, int32_t* tri_idx, int cap, int* n_tri);

/* The same triangle list, for callers that walk through the frames of a sequence one call at a time (morph_images() once per
 * frame, reference src/poppy.hpp:215): the point-location walks of the calling thread's previous call predict this call's
 * (each predicted step is verified, so the result never depends on the prediction); ~1.6x faster between neighbouring frames. */
int poppy_host_triangulate_next(const float* pts_xy, int n, int width, int height, int32_t* tri_idx, int cap, int* n_tri);

/* shape/mask ratio of frame j of an n_frames segment, reference src/poppy.hpp:181-210 with phase < 0:
 * 0 for j == 0, 1/(N-j) afterwards, capped at 1. */
double poppy_host_chain_ratio(int j, int n_frames);

/* Topology plan of a whole sequence: morphed points and triangle lists of every frame, computed on `threads`
 * host threads (0 = hardware concurrency).
 * chain == 0: frame f lerps (pts1, pts2) with shape_ratio[f]  (direct mode)
 * chain == 1: frame f lerps (morphed points of frame f-1, pts2) with shape_ratio[f]  (src/poppy.hpp:178-179) */
int poppy_host_plan_create(poppy_host_plan** out, const float* pts1_xy, const float* pts2_xy, int n, int width,
                           int height, int n_frames, const float* shape_ratio, int chain, int threads);
int poppy_host_plan_triangles(const poppy_host_plan* plan, const int32_t** tri_idx, const int32_t** tri_offsets,
                              int* max_triangles);
int poppy_host_plan_points(const poppy_host_plan* plan, int frame, const float** xy);
void poppy_host_plan_destroy(poppy_host_plan* plan);

/* C flavour of poppy::morph_images(): one frame, host buffers in and out. The context must have been created for
 * the same frame size; pyramid_levels is the context's (Settings::pyramid_levels at creation).
 * dst_bgr (rows `dst_step` bytes apart) and morphed_xy (n x 2) receive the outputs. Always returns 0.0 in the
 * reference; here 0 / negative status. */
int poppy_morph_images(poppy_cuda_ctx* ctx, const uint8_t* corrected1, size_t step1, const uint8_t* corrected2,
                       size_t step2, const float* gabor2, size_t gstep, const float* src_points1_xy,
                       const float* src_points2_xy, int n, double shape_ratio, double mask_ratio, uint8_t* dst_bgr,
                       size_t dst_step, float* morphed_xy);

/* ---- writer hand-off (reference src/poppy.hpp:219 `output.write(morphed)`; cv::VideoWriter src/poppy.cpp:249) -----------
 * A ring of page-locked frame buffers between the GPU frame ring and the caller's encoder. submit() enqueues the download
 * of rendered ring slots and returns (it only blocks while all `ring_frames` buffers are in flight); a delivery thread
 * waits for each copy and calls `write` strictly in frame order; with workers > 0 a thread pool first runs `convert` on
 * each frame (in place, any order). `write` / `convert` receive the frame index, the BGR pixels and their row stride. */
typedef struct poppy_host_writer poppy_host_writer;
typedef void (*poppy_write_fn)(void* user, int frame_index, uint8_t* bgr, int width, int height, size_t step);
int poppy_host_writer_create(poppy_host_writer** out, poppy_cuda_ctx* ctx, int ring_frames, poppy_write_fn write,
                             poppy_write_fn convert /* may be NULL */, int workers, void* user);
/* frames of ring slots [first_slot, first_slot + count) become frames first_frame_index.. of the output sequence */
int poppy_host_writer_submit(poppy_host_writer* w, int first_slot, int count, int first_frame_index);
int poppy_host_writer_flush(poppy_host_writer* w);          /* returns once every submitted frame has been written */
void poppy_host_writer_destroy_cuda(poppy_host_writer* w);  /* flushes, joins the threads, frees the ring */
/* The same ring delivering I420 frames (poppy_cuda_download_i420_async: converted on the GPU, W*H*3/2 bytes per buffer), the
 * pixel format of encoders fed yuv420p. `write` / `convert` receive a pointer to the Y plane with step = W; the U plane follows
 * at +W*H and the V plane at +W*H*5/4, (W/2) x (H/2) bytes each with rows of W/2 bytes. POPPY_CUDA_ERR_INVALID for an odd frame
 * size. Destroy it with poppy_host_writer_destroy_cuda. */
int poppy_host_writer_create_i420(poppy_host_writer** out, poppy_cuda_ctx* ctx, int ring_frames, poppy_write_fn write,
                                  poppy_write_fn convert /* may be NULL */, int workers, void* user);
/* The same ring delivering FFV1 packets (poppy_cuda_download_ffv1, encoded on the GPU): `packet` receives the frame index
 * and the packet's bytes, in frame order. Destroy it with poppy_host_writer_destroy_cuda. */
typedef void (*poppy_packet_fn)(void* user, int frame_index, const uint8_t* data, size_t size);
int poppy_host_writer_create_ffv1(poppy_host_writer** out, poppy_cuda_ctx* ctx, int ring_frames, poppy_packet_fn packet, void* user);

/* ---- FFV1 in Matroska (the reference's default output, cv::VideoWriter with fourcc FFV1) ------------------------------
 * poppy_host_ffv1_config: the configuration record (codec extradata) of the packets poppy_cuda_download_ffv1 writes at
 * width x height; *size receives its length, and POPPY_CUDA_ERR_INVALID is returned if dst is null or cap is smaller.
 * poppy_host_mkv_*: one video track (CodecID V_FFV1, CodecPrivate = that record) at fps_num / fps_den frames per second;
 * write() appends one packet as a keyframe SimpleBlock, close() writes the sizes and the duration and frees the writer.
 * Every call returns 0 or POPPY_CUDA_ERR_INVALID (bad argument, or the file could not be written). */
int poppy_host_ffv1_config(int width, int height, uint8_t* dst, size_t cap, size_t* size);
typedef struct poppy_host_mkv poppy_host_mkv;
int poppy_host_mkv_open(poppy_host_mkv** out, const char* path, int width, int height, int fps_num, int fps_den);
int poppy_host_mkv_write(poppy_host_mkv* m, const uint8_t* packet, size_t size);
int poppy_host_mkv_close(poppy_host_mkv* m);

/* The same machinery over a caller-supplied transport (tests run it without a GPU; another source of frames can reuse it). */
typedef struct poppy_host_writer_io {
    void* user;
    int (*download)(void* user, int slot, uint8_t* dst, size_t step, uint64_t* ticket);   /* start copying a slot */
    int (*wait)(void* user, uint64_t ticket);                                             /* may be NULL: copies are synchronous */
    int (*alloc)(void* user, size_t bytes, void** out);
    void (*release)(void* user, void* p);
    void (*write)(void* user, int frame_index, uint8_t* bgr, int width, int height, size_t step);
    void (*convert)(void* user, int frame_index, uint8_t* bgr, int width, int height, size_t step);   /* may be NULL */
    void* owned_transport;                                                                /* internal */
} poppy_host_writer_io;
int poppy_host_writer_create_io(poppy_host_writer** out, const poppy_host_writer_io* io, int width, int height, int ring_frames,
                                int workers);
void poppy_host_writer_destroy(poppy_host_writer* w);

/* The C++ shim (poppy_b200/csrc/host/morph_images.hpp: poppy::Settings, poppy::morph_images, poppy::morph_sequence with
 * the reference's argument order and semantics) behind C entry points, for callers and tests without a C++ toolchain:
 * the shim keeps its own device context per GPU (for the last frame size / pyramid levels), runs the host stages and, for
 * a sequence, the sliced chain render + writer ring; `write` receives the frames in order (reference src/poppy.hpp:177-243).
 * poppy_shim_morph_sequence takes gabor2 == NULL (gstep ignored): gabor2 is then derived on the device from corrected2, as
 * poppy::morph() derives it before its frame loop (src/poppy.hpp:119-122; poppy_cuda_set_pair). The per-frame entry points
 * keep requiring gabor2, as the reference's morph_images() does. */
int poppy_shim_morph_images(int width, int height, int pyramid_levels, const uint8_t* corrected1, size_t step1,
                            const uint8_t* corrected2, size_t step2, const float* gabor2, size_t gstep,
                            const float* src_points1_xy, const float* src_points2_xy, int n, double shape_ratio,
                            double mask_ratio, uint8_t* dst_bgr, size_t dst_step, float* morphed_xy);
int poppy_shim_morph_sequence(int width, int height, int pyramid_levels, const uint8_t* corrected1, size_t step1,
                              const uint8_t* corrected2, size_t step2, const float* gabor2, size_t gstep,
                              const float* src_points1_xy, const float* src_points2_xy, int n, int number_of_frames,
                              poppy_write_fn write, void* user);
/* The segments of a multi-image sequence (reference run(), src/poppy.cpp:266-328): segment i morphs one consecutive pair as
 * poppy_shim_morph_sequence does, and all segments (same frame size) are rendered together. `write` receives the
 * n_segments * number_of_frames frames in the reference's order: every frame of segment 0, then of segment 1, ... */
typedef struct poppy_shim_segment {
    const uint8_t* corrected1;
    size_t step1;
    const uint8_t* corrected2;
    size_t step2;
    const float* gabor2;          /* NULL: derived on the device from corrected2 */
    size_t gstep;
    const float* pts1_xy;
    const float* pts2_xy;
    int n;
} poppy_shim_segment;
int poppy_shim_morph_segments(int width, int height, int pyramid_levels, const poppy_shim_segment* segments, int n_segments,
                              int number_of_frames, poppy_write_fn write, void* user);
/* The same on several GPUs of one box: the segments are sharded over the first G = min(n_devices, n_segments) entries of
 * `devices`, devices[g] rendering segments [g * K / G, (g + 1) * K / G) on its own context and host thread (the others stay
 * idle). The frames and the order of the `write` calls equal poppy_shim_morph_segments's; `write` is called from a library
 * thread, one call at a time. Before anything is planned or rendered: POPPY_CUDA_ERR_INVALID for devices == NULL,
 * n_devices < 1, a duplicate or a negative index, then POPPY_CUDA_ERR_NO_DEVICE without a GPU, then POPPY_CUDA_ERR_INVALID
 * for an index >= poppy_cuda_device_count(). */
int poppy_shim_morph_segments_devices(const int* devices, int n_devices, int width, int height, int pyramid_levels,
                                      const poppy_shim_segment* segments, int n_segments, int number_of_frames, poppy_write_fn write,
                                      void* user);
void poppy_shim_release(void);            /* frees the shim's cached contexts, one per device used */

const char* poppy_host_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* POPPY_HOST_H_ */
