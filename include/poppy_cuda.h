/* poppy_cuda.h — C ABI of the B200 (sm_100a) morph renderer.
 *
 * This is the device boundary of the drop-in for the reference's per-frame morph path. The reference has no
 * FFI for this path: the boundary there is the in-process C++ call
 *     double poppy::morph_images(...)                       (reference src/algo.hpp:26, src/algo.cpp:178-273)
 * configured by poppy::Settings::pyramid_levels             (reference src/settings.hpp:20, read at algo.cpp:261)
 * and driven by the frame loop of poppy::morph<Twriter>()   (reference src/poppy.hpp:177-243).
 * The retained C++ host shim (poppy_b200/csrc/host/morph_images.hpp, same signature semantics) performs the host
 * stages (clip_points / make_uniq / Delaunay topology / vertex index lookup, reference src/algo.cpp:184-213)
 * and calls the functions below for everything from morph_points() to the final 8-bit frame
 * (reference src/algo.cpp:202, 216-265; src/blend.hpp:11-91; src/util.cpp:113-148).
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a negative
 * poppy_cuda_status; no C++ exception crosses this line; there is NO CPU fallback — without a CUDA device
 * poppy_cuda_create fails with POPPY_CUDA_ERR_NO_DEVICE. One context per GPU, driven by one host thread;
 * calls on distinct contexts are thread-safe. Host buffers are caller-owned (pinned memory makes the copies
 * asynchronous); all device memory is owned by the context.
 */
#ifndef POPPY_CUDA_H_
#define POPPY_CUDA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct poppy_cuda_ctx poppy_cuda_ctx;

typedef enum poppy_cuda_status {
    POPPY_CUDA_OK = 0,
    POPPY_CUDA_ERR_NO_DEVICE = -1,   /* no CUDA device / driver: the path does not run */
    POPPY_CUDA_ERR_INVALID = -2,     /* bad argument (null pointer, size out of range, index out of range) */
    POPPY_CUDA_ERR_CAPACITY = -3,    /* more points / triangles / frames than the context was created for */
    POPPY_CUDA_ERR_STATE = -4,       /* call sequence error (render before set_pair / set_points, ...) */
    POPPY_CUDA_ERR_CUDA = -5         /* a CUDA runtime call failed; see poppy_cuda_last_error */
} poppy_cuda_status;

/* Stage buffers that poppy_cuda_debug_read can fetch (context created with keep_stages != 0).
 * They are the stage boundaries of reference src/algo.cpp:202-265 (SURVEY.md section 3.2). Stages 0-7 belong to the last
 * rendered frame; POPPY_STAGE_MASK_BASIS belongs to the current pair and ignores `frame`. */
typedef enum poppy_cuda_stage {
    POPPY_STAGE_MORPHED_POINTS = 0,  /* n x 2 float            morph_points + clip_points, algo.cpp:202-205      */
    POPPY_STAGE_TRI_MAP = 1,         /* h x w int32            paint_triangles, algo.cpp:222-223                 */
    POPPY_STAGE_INV_M1 = 2,          /* T x 9 float            inv(morphHom1[k]) as create_map applies it, :154-157 */
    POPPY_STAGE_INV_M2 = 3,          /* T x 9 float            inv(morphHom2[k])                                  */
    POPPY_STAGE_WARPED1 = 4,         /* h x w x 3 uint8        remap(corrected1), algo.cpp:233                    */
    POPPY_STAGE_WARPED2 = 5,         /* h x w x 3 uint8        remap(corrected2), algo.cpp:238                    */
    POPPY_STAGE_MASK = 6,            /* h x w float            lbmask, algo.cpp:250-258                           */
    POPPY_STAGE_LAP_BLEND = 7,       /* h x w x 3 float (BGR interleaved)  LaplacianBlending::blend(), :261-262   */
    POPPY_STAGE_MASK_BASIS = 8       /* h x w float            m2 = 1 - gray(gabor2) of the current pair, :250-252  */
} poppy_cuda_stage;

int poppy_cuda_device_count(void);

/* width/height: frame size (both < 32767, as cv::remap requires). pyramid_levels: Settings::pyramid_levels
 * (any value >= 1; levels past 1x1 stay 1x1 exactly as cv::pyrDown/pyrUp do). max_points / max_triangles /
 * max_batch_frames bound set_points, render and the HBM frame ring. */
int poppy_cuda_create(poppy_cuda_ctx** out, int device, int width, int height, int pyramid_levels, int max_points,
                      int max_triangles, int max_batch_frames);
void poppy_cuda_destroy(poppy_cuda_ctx* ctx);

/* Geometry and capacities the context was created with (any pointer may be NULL). */
int poppy_cuda_get_info(const poppy_cuda_ctx* ctx, int* width, int* height, int* pyramid_levels, int* max_points,
                        int* max_triangles, int* max_batch_frames);

/* Options; call before the first render. */
int poppy_cuda_set_keep_stages(poppy_cuda_ctx* ctx, int keep);       /* 1: chunk size 1, stage buffers readable */
int poppy_cuda_set_chunk_frames(poppy_cuda_ctx* ctx, int frames);    /* frames rendered per kernel batch (>=1) */
int poppy_cuda_set_stage_timing(poppy_cuda_ctx* ctx, int enable);    /* CUDA-event timing per kernel class */
/* unsharp_mask stage (reference src/util.cpp:113-148, called at src/algo.cpp:263-264): two bit-identical routes.
 * Calm route: the level-0 collapse stores the 8-bit frame itself, and the exact GaussianBlur + medianBlur + threshold path
 * runs only on the strip chunks where a bound on |x - blur| (second differences of the stored bytes) does not rule out the
 * 0.3 norm threshold; everywhere else unsharp_mask() provably returns x. Dense route: the exact path on every pixel.
 * mode 0 (default): adaptive - calm route while few chunks of recent frames needed the exact path, dense route otherwise;
 * mode 1: dense always; mode 2: calm route always. */
int poppy_cuda_set_unsharp_mode(poppy_cuda_ctx* ctx, int mode);
/* Strip chunks (120 columns x 24 rows of a frame) that took the exact unsharp path / all chunks, since the last call;
 * syncs. */
int poppy_cuda_unsharp_stats(poppy_cuda_ctx* ctx, uint64_t* chunks_exact, uint64_t* chunks_total);
/* Capacity (entries per frame) of the per-tile triangle lists that feed the rasteriser. The default suits any
 * Delaunay mesh; a frame whose lists do not fit is still rendered exactly (every tile then tests every triangle of
 * that frame), only slower. Exposed so that this path can be exercised by the tests. */
int poppy_cuda_set_tile_list_capacity(poppy_cuda_ctx* ctx, int entries_per_frame);

/* corrected1 / corrected2 (8UC3 BGR, row stride in bytes) and gabor2 (32FC3 BGR in [0,1], row stride in bytes) of
 * one image pair: the Mat arguments of morph_images (reference src/algo.cpp:178). H2D once per pair.
 * gabor2_bgr32f == NULL: the context derives what it needs of gabor2 on the device from corrected2, as poppy::morph()
 * derives gabor2 before its frame loop (gabor_filter(corrected2 * 1/255) with the default parameters, reference
 * src/poppy.hpp:119-122; set_image selector 3). Only corrected1 and corrected2 cross PCIe, and the mask basis is
 * bit-identical to the one set_pair makes from poppy_cuda_gabor_filter(corrected2 * float(1/255.0)). */
int poppy_cuda_set_pair(poppy_cuda_ctx* ctx, const uint8_t* bgr1, size_t step1, const uint8_t* bgr2, size_t step2,
                        const float* gabor2_bgr32f, size_t gstep);

/* One image of the pair: which = 0 corrected1 (8UC3), 1 corrected2 (8UC3), 2 gabor2 (32FC3), 3 corrected2 (8UC3) with
 * the mask basis derived from it instead of a gabor2 (see poppy_cuda_set_pair; sets images 1 and 2). Lets a per-frame
 * caller re-upload only what changed between two morph_images() calls (in the reference's frame loop only corrected1
 * does, src/poppy.hpp:217). Asynchronous for pinned memory: poppy_cuda_sync() before the buffer is modified. The first
 * selector-3 call on a device also uploads the filter taps and waits for that copy. Device staging is allocated on first
 * use: 3 bytes per pixel for selectors 0, 1 and 3, 12 for selector 2. */
int poppy_cuda_set_image(poppy_cuda_ctx* ctx, int which, const void* data, size_t step);
/* corrected1 := rendered frame `slot` of the ring, device to device: the `corrected1 = morphed.clone()` of the reference
 * frame loop (src/poppy.hpp:217) for callers that drive the recurrence one render call per frame. */
int poppy_cuda_set_source1_from_slot(poppy_cuda_ctx* ctx, int slot);

/* srcPoints1 / srcPoints2 (n x 2 float, x then y), unclipped as the caller holds them. n < 3 is allowed (no triangles:
 * the frame is the blend of the unwarped pair, as in the reference). */
int poppy_cuda_set_points(poppy_cuda_ctx* ctx, const float* pts1_xy, const float* pts2_xy, int n);

/* Render n_frames frames into the HBM frame ring (slots 0 .. n_frames-1).
 * shape_ratio[f], mask_ratio[f]: the shapeRatio / maskRatio arguments of morph_images for frame f.
 * tri_idx: concatenated triangle vertex indices (3 per triangle, indices into the point sets) of every frame's
 * Delaunay mesh of the *morphed* points, in cv::Subdiv2D::getTriangleList order (this order decides which
 * triangle wins a shared pixel, reference src/algo.cpp:95-106); tri_offsets[f] .. tri_offsets[f+1] delimit frame f
 * (in triangles).
 * chain == 0: every frame is rendered from the pair and point sets as uploaded (direct mode; the reference's
 *             "-f 1 -p s" frame, src/poppy.hpp:186-200).
 * chain == 1: frame f>0 takes frame f-1's output as corrected1 and frame f-1's morphed points as srcPoints1
 *             (the recurrence of the reference frame loop, src/poppy.hpp:178-179,217-218).
 * Asynchronous with respect to the device; host arrays are consumed before the call returns. */
int poppy_cuda_render(poppy_cuda_ctx* ctx, int n_frames, const float* shape_ratio, const double* mask_ratio,
                      const int32_t* tri_idx, const int32_t* tri_offsets, int chain);

/* Same, into ring slots [first_slot, first_slot + n_frames): frame i of the call (arrays indexed from 0) lands in slot
 * first_slot + i. Lets a caller stream a long sequence through the ring slice by slice - plan slice k+1 on the host
 * while slice k renders and slice k-1 downloads (the frame loop of src/poppy.hpp:172-243 with the writer hand-off
 * overlapped). With chain == 1 and first_slot > 0 the call continues the chain of the previous call, which must have ended
 * at slot first_slot - 1 (a long chain rendered slice by slice). */
int poppy_cuda_render_range(poppy_cuda_ctx* ctx, int first_slot, int n_frames, const float* shape_ratio,
                            const double* mask_ratio, const int32_t* tri_idx, const int32_t* tri_offsets, int chain);

/* Resident plan: the packed triangle lists of a whole sequence (the layout poppy_cuda_render takes) copied to HBM and
 * validated once, after poppy_cuda_set_points. poppy_cuda_render_planned then renders plan frames
 * [plan_first, plan_first + n_frames) into ring slots first_slot.. with shape_ratio / mask_ratio indexed from 0 for the call -
 * no per-render staging of the lists (at 4K / 20k points they are 290 MB per 600 frames). A new point set invalidates the plan. */
int poppy_cuda_set_plan(poppy_cuda_ctx* ctx, const int32_t* tri_idx, const int32_t* tri_offsets, int n_frames);
int poppy_cuda_render_planned(poppy_cuda_ctx* ctx, int first_slot, int plan_first, int n_frames, const float* shape_ratio,
                              const double* mask_ratio, int chain);

/* ---- segments of a multi-image sequence ---------------------------------------------------------------------------------
 * The reference's run() (src/poppy.cpp:266-328) morphs each consecutive pair of a list of images as one segment: a chain of
 * number_of_frames frames (src/poppy.hpp:177-243). Segments have the same frame size and depend on no rendered frame of
 * each other, so they can be rendered together: a kernel batch holds step j of up to chunk-frames segments, and the
 * launches per step do not grow with the number of segments. This state lives beside the single pair and leaves it,
 * the points and the resident plan as they are.
 *
 * poppy_cuda_set_segments: room for n_segments segments (each with its own corrected1, corrected2, chain source, mask
 * basis and point sets in HBM) and a ring window of `window` slots per segment: step j of segment s lands in ring slot
 * s * window + j % window. window >= 2 (step j reads step j-1's points); n_segments * window <= max_batch_frames
 * (POPPY_CUDA_ERR_CAPACITY). Replaces any earlier segments.
 * poppy_cuda_set_segment: poppy_cuda_set_pair + poppy_cuda_set_points for segment s (gabor2 == NULL: the mask basis is
 * derived from corrected2 on the device); n <= max_points. Synchronous. */
int poppy_cuda_set_segments(poppy_cuda_ctx* ctx, int n_segments, int window);
int poppy_cuda_set_segment(poppy_cuda_ctx* ctx, int s, const uint8_t* bgr1, size_t step1, const uint8_t* bgr2, size_t step2,
                           const float* gabor2_bgr32f, size_t gstep, const float* pts1_xy, const float* pts2_xy, int n);
/* Render steps [first_step, first_step + n_steps) of every segment as chains (frame j from frame j-1 and its morphed
 * points). shape_ratio / mask_ratio: one entry per step, indexed from 0 for the call. tri_offsets has n_steps * K + 1
 * entries: the list of step first_step + r of segment s is entry r * K + s (step-major), with vertex indices into that
 * segment's points (checked against its own n). A call with first_step > 0 continues where the previous segment render
 * ended (POPPY_CUDA_ERR_STATE otherwise); every segment must have been set. Segments go in groups of at most chunk-frames
 * segments; all steps of a group run on one render lane and the groups go round-robin over the lanes. Not on keep_stages
 * contexts. Frames are read with the slot-based calls (download, checksum, frame_device_ptr); poppy_cuda_last_render_ms
 * times the call. A pair render afterwards ends the segment render (and a segment render a sliced pair chain). */
int poppy_cuda_render_segments(poppy_cuda_ctx* ctx, int first_step, int n_steps, const float* shape_ratio,
                               const double* mask_ratio, const int32_t* tri_idx, const int32_t* tri_offsets);
/* morphedPoints of step `step` of segment s (its own n x 2 float), while the step is still in the segment's window. */
int poppy_cuda_get_segment_points(poppy_cuda_ctx* ctx, int s, int step, float* xy);

/* Copy frames [first, first+count) (8UC3 BGR) to host memory: row stride `step` bytes, `frame_stride` bytes
 * between frames. Ordered after every render queued so far, on a separate copy stream (renders of other slots are not
 * held up; a render of slots with a download pending waits for it). Asynchronous if dst is pinned;
 * poppy_cuda_sync() before reading. */
int poppy_cuda_download(poppy_cuda_ctx* ctx, int first, int count, uint8_t* dst, size_t step, size_t frame_stride);

/* poppy_cuda_download that also returns a ticket; poppy_cuda_download_wait(ticket) blocks until that copy (and every earlier
 * one) has landed, without waiting for renders or later downloads. wait may be called from another host thread (the writer
 * hand-off, include/poppy_host.h). At most 64 tickets may be outstanding. */
int poppy_cuda_download_async(poppy_cuda_ctx* ctx, int first, int count, uint8_t* dst, size_t step, size_t frame_stride,
                              uint64_t* ticket);
int poppy_cuda_download_wait(poppy_cuda_ctx* ctx, uint64_t ticket);

/* Frames [first, first+count) as I420 (YUV 4:2:0, BT.601 limited range), byte for byte what
 * cv::cvtColor(bgr, out, COLOR_BGR2YUV_I420) gives for the BGR frame: per frame the Y plane (W x H), then U and V ((W/2) x (H/2)
 * each), every row tightly packed, W*H*3/2 bytes; frame i lands at dst + i * frame_stride. Chroma is the top-left pixel of each
 * 2 x 2 block. The conversion runs on the device, so half the bytes of a BGR download cross PCIe. Ordering is that of
 * poppy_cuda_download: the conversion and the copies run on the copy stream after every render queued so far, and a later
 * render of these slots waits for both. Device staging of a few frames is allocated on the first call; a larger count goes
 * through it in pieces. POPPY_CUDA_ERR_INVALID for an odd W or H (cv::cvtColor throws there too), a null dst, a bad range or
 * frame_stride < W*H*3/2. Asynchronous if dst is pinned; poppy_cuda_sync() before reading. The _async flavour returns a ticket
 * of the same pool as poppy_cuda_download_async, for poppy_cuda_download_wait. */
int poppy_cuda_download_i420(poppy_cuda_ctx* ctx, int first, int count, uint8_t* dst, size_t frame_stride);
int poppy_cuda_download_i420_async(poppy_cuda_ctx* ctx, int first, int count, uint8_t* dst, size_t frame_stride, uint64_t* ticket);
/* Frames [first, first+count) as lossless FFV1 packets, encoded on the device: FFV1 version 3 with the range coder, RGB
 * (JPEG2000-RCT), 8 bits, no alpha, every frame a keyframe, a slice grid that depends on the frame size only
 * (poppy_host_ffv1_config gives the matching configuration record). The packets land back to back at dst; sizes[i] receives
 * the size of packet i. Only the packet bytes and the sizes cross PCIe. The bytes are a function of the frame alone. Ordering
 * is that of poppy_cuda_download: encoding and copies run on the copy stream after every render queued so far, and a later
 * render of these slots waits for them; the call returns when dst and sizes are filled. Device staging is allocated on the
 * first call. POPPY_CUDA_ERR_INVALID for a null dst or sizes or a bad range, and when the packets need more than `cap`
 * bytes: sizes[] is still filled then, so their sum is the capacity to pass. */
int poppy_cuda_download_ffv1(poppy_cuda_ctx* ctx, int first, int count, uint8_t* dst, size_t cap, uint32_t* sizes);
/* Page-locked host memory for download targets (asynchronous copies need it). */
int poppy_cuda_alloc_pinned(size_t bytes, void** out);
void poppy_cuda_free_pinned(void* p);

/* morphedPoints of frame `frame` of the last render (n x 2 float) — the out-parameter of morph_images. */
int poppy_cuda_get_morphed_points(poppy_cuda_ctx* ctx, int frame, float* xy);

/* Device address of frame slot `frame` (8UC3, tightly packed rows) for zero-copy consumers; *bytes = frame size. */
int poppy_cuda_frame_device_ptr(poppy_cuda_ctx* ctx, int frame, void** dptr, size_t* bytes);

/* 64-bit FNV-1a style checksum of frames [first, first+count) computed on the device (order dependent). */
int poppy_cuda_checksum(poppy_cuda_ctx* ctx, int first, int count, uint64_t* out);

int poppy_cuda_sync(poppy_cuda_ctx* ctx);

/* The CUDA stream every launch of this context goes to (cudaStream_t), for event timing by the caller. */
int poppy_cuda_get_stream(poppy_cuda_ctx* ctx, void** stream);

/* Device time (ms, CUDA events on the context's stream) of the last poppy_cuda_render call; syncs. */
int poppy_cuda_last_render_ms(poppy_cuda_ctx* ctx, float* ms);

/* Kernel launches issued by this context since creation (its own kernels only, memsets/copies not counted). */
int poppy_cuda_launch_count(poppy_cuda_ctx* ctx, uint64_t* launches);

/* Per-kernel-class device time of the last render (stage timing enabled); "misc" also adds the mask-basis filter launches
 * of set_image selector 3 since then. Fills up to `cap` entries; returns the number of classes. names[i] points to a static
 * string. */
int poppy_cuda_stage_times(poppy_cuda_ctx* ctx, const char** names, float* ms, uint64_t* launches, int cap);

/* Fetch a stage buffer of frame `frame` of the last render (keep_stages contexts only). `bytes` must match. */
int poppy_cuda_debug_read(poppy_cuda_ctx* ctx, int stage, int frame, void* dst, size_t bytes);

/* Last error text of this context (or of the failed create when ctx == NULL). */
const char* poppy_cuda_last_error(const poppy_cuda_ctx* ctx);

/* Build identification: "poppy_cuda <version> sm_100a". */
const char* poppy_cuda_version(void);

/* ---- input conditioning ahead of the path (SURVEY.md 8(f-3)) ----------------------------------------------------------
 * poppy::blur_margin(src, szUnion, dst), reference src/util.cpp:574-602: the 8-bit BGR source centred on a black
 * union_w x union_h canvas whose four margins are blurred by cv::GaussianBlur(127 x 127, sigma 6) (OpenCV's fixed-point
 * 8-bit path, reproduced exactly). Stand-alone (no context): runs on `device`, fails with POPPY_CUDA_ERR_NO_DEVICE without
 * one and with POPPY_CUDA_ERR_INVALID where the reference's cv::Mat ROI assertions would throw. */
int poppy_cuda_blur_margin(int device, const uint8_t* src, size_t src_step, int cols, int rows, int union_w, int union_h,
                           uint8_t* dst, size_t dst_step);
const char* poppy_cuda_blur_margin_last_error(void);      /* of the calling thread's last blur_margin / gabor_filter / denoise call */

/* poppy::gabor_filter(src, dst) with the reference's defaults (src/util.cpp:40-60, src/util.hpp:95, called at
 * src/poppy.hpp:122): src / dst are float BGR (rows x cols x 3), dst = mean over 16 orientations of the clamped 13 x 13 Gabor
 * responses. cv::filter2D evaluates these by a double-precision block DFT; this entry point sums the same correlation directly
 * in double, so results agree to the float rounding of a value known to ~1e-15: floating-point parity with tolerance
 * (|diff| <= 1.2e-7 everywhere; on textured images at most 20 values per million differ by more than the DFT's own round-off
 * around zero, 1e-12; tests/test_margin.py), not bit-exact. */
int poppy_cuda_gabor_filter(int device, const float* src, size_t src_step, int cols, int rows, float* dst, size_t dst_step);

/* cv::fastNlMeansDenoising(src, dst, h, template_window_size, search_window_size) of an 8-bit BGR image (NORM_L2), as the
 * reference's run() calls it under --denoise (src/poppy.cpp:172, 269-311), reproduced bit for bit: the weight table is built
 * on the host with std::exp as OpenCV builds it, and every per-pixel step is exact integer arithmetic. OpenCV's defaults are
 * h = 3, 7, 21; even window sizes round up to the next odd size, and only h * h counts. Stand-alone (no context), host
 * input and output (src_step / dst_step: row strides in bytes); dst may equal src. Supported range, after rounding:
 * template_window_size <= 15 and search_window_size <= 63. POPPY_CUDA_ERR_INVALID for a null pointer, cols or rows < 1,
 * a step below cols * 3, a window size < 1 or beyond that range, or a non-finite h; POPPY_CUDA_ERR_NO_DEVICE without a
 * GPU. Error text: poppy_cuda_blur_margin_last_error(). */
int poppy_cuda_denoise(int device, const uint8_t* src, size_t src_step, int cols, int rows, float h, int template_window_size,
                       int search_window_size, uint8_t* dst, size_t dst_step);

#ifdef __cplusplus
}
#endif
#endif /* POPPY_CUDA_H_ */
