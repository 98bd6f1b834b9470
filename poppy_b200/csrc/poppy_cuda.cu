// poppy_cuda.cu — context, HBM layout and the extern "C" layer declared in include/poppy_cuda.h.
//
// HBM layout per context (W x H frame, L pyramid levels, chunk of B frames in flight):
//   pair (resident)   : src1, src2 as BGRX uchar4 [H][W]; mask basis m2 float [H][pitch0]; clipped point sets
//                       (pitch0 = W rounded up to 32 elements: rows of every per-pixel plane start 128-byte aligned)
//   frame ring        : max_batch_frames x [H][W*3] 8-bit BGR — the rendered frames stay in HBM until downloaded
//   morphed points    : max_batch_frames x max_points float2
//   chunk scratch (xB): FrameParams; triangle indices; TriInverse / TriRaster records; triangle-ID map int32 [H][W];
//                       warped pair 2 x uint32 BGRX [H][pitch0]; Gaussian levels 1..L (7 planes); collapsed levels 0..L
//                       (3 planes); level-0 blend mask float [H][pitch0]
//   I420 staging      : (optional, poppy_cuda_download_i420) up to kI420StageFrames x W*H*3/2 bytes, allocated on first use
//   FFV1 staging      : (optional, poppy_cuda_download_ffv1) a piece of up to kFfv1StagePixels pixels: 12 B of symbols and
//                       3 B + slice allowance of slice slots per pixel, the packets, per-slice tables; overflow scratch
//                       on demand. Allocated on first use.
//   segments (optional, poppy_cuda_set_segments): per segment the pair's resident data - corrected1, corrected2 and chain
//                       arrays, a mask basis (one allocation, padded_pixels() floats each), raw and clipped point sets;
//                       per lane a SegFrame table and a BGRX staging plane per frame of a chunk
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/poppy_cuda.h"
#include "device/kernels.cuh"
#include "ffv1_format.hpp"

using namespace poppy;

namespace {

thread_local std::string g_create_error;

enum KernelClass { KC_POINTS = 0, KC_GEOMETRY, KC_BIN, KC_WARP, KC_PYR_DOWN, KC_COLLAPSE, KC_CALM, KC_UNSHARP, KC_MISC, KC_COUNT };
const char* const kClassNames[KC_COUNT] = {"lerp_points", "tri_geometry", "bin_triangles", "raster_warp",
                                           "pyr_down", "blend_collapse", "calm_analysis", "unsharp_store", "misc"};

struct TimedLaunch { int cls; cudaEvent_t a, b; };

// Adaptive routing of the unsharp stage (unsharp_mode 0): calm route while at most this share of the strip chunks of recent
// frames needed (or, on the dense route, would have needed) the exact path; the dense route otherwise. On the dense route
// every kCalmProbeEvery-th chunk also runs the calm analysis on its finished frames - a few percent of a chunk's time - so
// that the router notices when the content calms down again. (Break-even: the calm route costs about half of the dense one
// plus 1.4x the dense cost of whatever it flags.)
constexpr double kCalmRouteMaxShare = 0.2;
constexpr unsigned kCalmProbeEvery = 8;      // on the dense route: every n-th chunk also runs the (cheap) byte scan for the statistic

// rows per CTA of the exact unsharp pass over flagged strip chunks (the dense pass used 216; a finer grain keeps calm
// regions out of the exact path at the price of the 10-row warm-up per chunk)
constexpr int kSparseChunkRows = 24;

// Render lanes: consecutive chunks of a direct-mode render go round-robin to the lanes. Measured at 4K: 1 lane 2,694,
// 2: 2,952, 3: 3,150, 4: 3,219-3,259, 8: 3,263 frames/s.
constexpr int kRenderLanes = 4;

// I420 downloads convert at most this many frames per piece into device staging (a 4K frame is 12.4 MB in I420)
constexpr int kI420StageFrames = 8;

// FFV1 downloads encode at most this many pixels per piece (8 4K frames, 1,003 MB of device staging)
constexpr size_t kFfv1StagePixels = (size_t)8 * 3840 * 2160;

}  // namespace

struct poppy_cuda_ctx {
    int device = 0, w = 0, h = 0, levels = 0, max_points = 0, max_tri = 0, max_frames = 0;
    int chunk = 0;            // frames per kernel batch (0 = not yet allocated)
    int want_chunk = 0;
    bool keep_stages = false, stage_timing = false;
    bool have_pair = false, have_points = false;
    bool have_image[3] = {false, false, false};
    uint8_t* d_stage_u8 = nullptr;       // upload staging of set_image, kept between calls
    float* d_stage_f32 = nullptr;        // only for a caller-supplied gabor2 (selector 2)
    int n_points = 0, last_frames = 0;
    int chain_next_slot = -1;            // ring slot at which a sliced chain render may continue (-1: no chain in progress)
    std::vector<cudaEvent_t> tickets;    // download tickets (poppy_cuda_download_async), indexed ticket % size
    uint64_t next_ticket = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    // downloads run on their own stream so that they overlap the render of other ring slots; a render that would
    // overwrite slots with a download pending waits for it
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_rendered = nullptr, ev_copied = nullptr;
    int copy_lo = 0, copy_hi = 0;        // ring slots [lo, hi) with a download enqueued since the last sync
    uint8_t* d_i420 = nullptr;           // I420 staging of poppy_cuda_download_i420 (copy stream only)
    int i420_frames = 0;                 // frames d_i420 holds
    struct Ffv1Stage {                   // poppy_cuda_download_ffv1 (copy stream only)
        int frames = 0, nh = 0, nv = 0;
        size_t cap = 0, scratch_cap = 0, scratch_slices = 0, packets_cap = 0;
        uint32_t* d_sym = nullptr;
        uint8_t *d_slots = nullptr, *d_packets = nullptr, *d_tables = nullptr, *d_scratch = nullptr;
        uint32_t *d_sizes = nullptr, *d_frame_sizes = nullptr;
        uint64_t* d_offsets = nullptr;
        int *d_slot_of = nullptr, *d_overflow = nullptr;   // d_overflow: count, then the list
        int* h_overflow = nullptr;                         // pinned
    } ffv1;
    std::string err;
    uint64_t launches = 0;

    std::vector<LevelDesc> lv;           // level 0 .. L
    std::vector<size_t> g_off, o_off;    // float offsets of level k inside d_g / d_o for ONE frame-chunk block
    size_t g_floats = 0, o_floats = 0;   // per chunk

    // resident
    uchar4* d_src_stage = nullptr;       // linear BGRX staging for the array uploads
    // sources as uchar4 CUDA arrays (texture gather) + point/border texture objects; index 2 = the chain source
    // (frame j-1 of a recurrence, reference src/poppy.hpp:178-179)
    cudaArray_t a_src[3] = {nullptr, nullptr, nullptr};
    cudaTextureObject_t t_src[3] = {0, 0, 0};
    float* d_mbasis = nullptr;
    float2 *d_pts1_raw = nullptr, *d_pts2_raw = nullptr, *d_pts1 = nullptr, *d_pts2 = nullptr, *d_morphed = nullptr;
    uint8_t* d_frames = nullptr;
    unsigned long long* d_sum = nullptr;
    // Chunk scratch of kRenderLanes lanes, each with its own stream: consecutive chunks of a direct-mode render go
    // round-robin to the lanes, so the issue-bound kernels of one chunk overlap the latency- and bandwidth-bound kernels of
    // the others.
    struct Lane {
        cudaStream_t stream = nullptr;
        cudaEvent_t ev_staged = nullptr, ev_done = nullptr;
        FrameParams* d_fp = nullptr;
        int3* d_tri = nullptr;
        TriInverse* d_inv = nullptr;
        TriRaster* d_rast = nullptr;
        int* d_trimap = nullptr;             // stage dumps only (keep_stages)
        int *d_tile_cnt = nullptr, *d_tile_off = nullptr, *d_tile_list = nullptr, *d_overflow = nullptr;
        uint32_t* d_warped = nullptr;        // per frame: remap of image 1, remap of image 2 (packed BGRX words)
        float *d_mask0 = nullptr, *d_g = nullptr, *d_o = nullptr;
        // calm analysis of the unsharp stage: clamp-excess flags of out[0], block / strip-chunk / collapse-tile flags
        unsigned char* d_excess = nullptr;
        unsigned char *d_block_dev = nullptr, *d_block_flags = nullptr, *d_chunk_flags = nullptr, *d_tile_flags = nullptr;
        int* d_calm_counts = nullptr;
        int* h_calm_counts = nullptr;        // pinned: flagged strip chunks per frame of the lane's last calm-route chunk
        cudaEvent_t ev_calm = nullptr;
        int calm_pending = 0;                // frames whose counts are on their way to h_calm_counts
        std::vector<CollapseMaps> maps;      // tensor maps of level k's collapse (index k)
        FrameParams* h_fp = nullptr;         // pinned staging
        int32_t* h_tri = nullptr;
        // segment renders: the chunk's per-frame sources (d_seg, pinned staging h_seg) and the BGRX staging of its frames
        // for the chain arrays, seg_cap frames each
        SegFrame *d_seg = nullptr, *h_seg = nullptr;
        uchar4* d_seg_stage = nullptr;
        int seg_cap = 0;
    } lane[kRenderLanes];
    int n_lanes = 0;                         // lanes allocated (0 = none yet)
    int n_tiles = 0, list_cap = 0;
    // levels tail_k0 .. L run in one launch (k_pyramid_tail); 0 = none (no level is small enough)
    int tail_k0 = 0;
    TailLevel* d_tail_levels = nullptr;
    // unsharp stage. Calm route: the fused level-0 collapse stores the frame and only the strip chunks that can reach the
    // unsharp threshold run the exact blur + median path. Dense route: level-0 collapse to float planes + the exact path on
    // every pixel. 0 = adaptive (the calm route while the share of flagged chunks seen on recent frames stays low, the dense
    // route otherwise, probing the calm route now and then); 1 = dense always (forced by keep_stages); 2 = calm always.
    int unsharp_mode = 0;
    double calm_share = 1.0;                 // running share of flagged strip chunks (starts pessimistic: dense until a scan says otherwise)
    unsigned route_tick = kCalmProbeEvery - 1;   // the first dense chunk carries a scan
    unsigned probe_every = kCalmProbeEvery;
    // resident plan (poppy_cuda_set_plan): the packed triangle lists of a whole sequence in HBM, validated once
    int3* d_plan_tri = nullptr;
    size_t plan_cap = 0;                     // triangles d_plan_tri holds
    std::vector<int32_t> plan_off;           // n + 1 offsets (triangles), plan_off[0] == 0
    int plan_points = -1;                    // n_points the plan was validated against      // backs off (x2, up to 64) while the scans keep reporting busy content
    int mm_pitch = 0;                        // blocks per row of the clamp-excess table, padded
    size_t mm_stride = 0;
    unsigned long long* d_calm_total = nullptr;      // flagged strip chunks since the last stats read
    unsigned long long* d_probe_total = nullptr;     // sink of the statistic-only scans
    uint64_t calm_chunks_total = 0, dense_chunks_total = 0;

    // Segments of a multi-image sequence (poppy_cuda_set_segments): independent chains of the same frame size, rendered
    // together. Step j of segment s lands in ring slot s * seg_window + j % seg_window.
    struct Segment {
        cudaArray_t a[3] = {nullptr, nullptr, nullptr};      // corrected1, corrected2, chain source (the previous step's frame)
        cudaTextureObject_t t[3] = {0, 0, 0};
        int n = 0;                                           // points
        bool set = false;
    };
    std::vector<Segment> seg;
    int seg_window = 0;
    int seg_next_step = -1;                  // step at which a segment render may continue (-1: none in progress)
    float* d_seg_basis = nullptr;            // n_seg x padded_pixels()
    float2 *d_seg_raw = nullptr, *d_seg_pts1 = nullptr, *d_seg_pts2 = nullptr;   // raw: 2 x max_points, clipped: max_points per segment

    std::vector<TimedLaunch> timed;
    std::vector<cudaEvent_t> event_pool;
    float class_ms[KC_COUNT] = {0};
    uint64_t class_launches[KC_COUNT] = {0};

    size_t frame_bytes() const { return (size_t)w * h * 3; }
    size_t pixels() const { return (size_t)w * h; }
    int pitch0() const { return lv[0].pitch; }
    size_t padded_pixels() const { return lv[0].plane_stride; }
};

namespace {

int fail(poppy_cuda_ctx* c, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf; else g_create_error = buf;
    return code;
}

#define CU_TRY(c, expr)                                                                                     \
    do {                                                                                                    \
        cudaError_t e_ = (expr);                                                                            \
        if (e_ != cudaSuccess)                                                                              \
            return fail((c), POPPY_CUDA_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

template <class T> cudaError_t dmalloc(T** p, size_t count) { return cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(T)); }

void free_chunk(poppy_cuda_ctx* c) {
    for (auto& l : c->lane) {
        cudaFree(l.d_fp); cudaFree(l.d_tri); cudaFree(l.d_inv); cudaFree(l.d_rast); cudaFree(l.d_trimap);
        cudaFree(l.d_tile_cnt); cudaFree(l.d_tile_off); cudaFree(l.d_tile_list); cudaFree(l.d_overflow);
        cudaFree(l.d_warped); cudaFree(l.d_mask0); cudaFree(l.d_g); cudaFree(l.d_o);
        cudaFree(l.d_excess); cudaFree(l.d_block_dev); cudaFree(l.d_block_flags); cudaFree(l.d_chunk_flags); cudaFree(l.d_tile_flags); cudaFree(l.d_calm_counts);
        cudaFreeHost(l.h_fp); cudaFreeHost(l.h_tri); cudaFreeHost(l.h_calm_counts);
        cudaFree(l.d_seg); cudaFreeHost(l.h_seg); cudaFree(l.d_seg_stage);
        cudaStream_t st = l.stream; cudaEvent_t e1 = l.ev_staged, e2 = l.ev_done, e3 = l.ev_calm;
        l = poppy_cuda_ctx::Lane();
        l.stream = st; l.ev_staged = e1; l.ev_done = e2; l.ev_calm = e3;
    }
    c->chunk = 0;
    c->n_lanes = 0;
}

void free_segments(poppy_cuda_ctx* c) {
    for (auto& S : c->seg)
        for (int i = 0; i < 3; ++i) {
            if (S.t[i]) cudaDestroyTextureObject(S.t[i]);
            if (S.a[i]) cudaFreeArray(S.a[i]);
        }
    c->seg.clear();
    cudaFree(c->d_seg_basis); cudaFree(c->d_seg_raw); cudaFree(c->d_seg_pts1); cudaFree(c->d_seg_pts2);
    c->d_seg_basis = nullptr; c->d_seg_raw = c->d_seg_pts1 = c->d_seg_pts2 = nullptr;
    c->seg_window = 0;
    c->seg_next_step = -1;
}

// uchar4 array with a point-sampled, border-addressed (zero) texture over it, as the pair's sources
cudaError_t make_source_array(int w, int h, cudaArray_t* a, cudaTextureObject_t* t) {
    const cudaChannelFormatDesc fmt = cudaCreateChannelDesc<uchar4>();
    cudaError_t e = cudaMallocArray(a, &fmt, (size_t)w, (size_t)h, cudaArrayTextureGather);
    if (e != cudaSuccess) return e;
    cudaResourceDesc res{};
    res.resType = cudaResourceTypeArray;
    res.res.array.array = *a;
    cudaTextureDesc td{};
    td.addressMode[0] = td.addressMode[1] = cudaAddressModeBorder;      // BORDER_CONSTANT(0)
    td.filterMode = cudaFilterModePoint;
    td.readMode = cudaReadModeElementType;
    td.normalizedCoords = 0;
    return cudaCreateTextureObject(t, &res, &td, nullptr);
}

// 8-bit BGR host image -> BGRX array, through the pair's upload staging on the context's stream
int upload_source(poppy_cuda_ctx* c, const uint8_t* data, size_t step, cudaArray_t dst) {
    const size_t row = (size_t)c->w * 3, trow = (size_t)c->w * 4;
    CU_TRY(c, cudaMemcpy2DAsync(c->d_stage_u8, row, data, step, row, c->h, cudaMemcpyHostToDevice, c->stream));
    launch_bgr_to_bgrx(c->stream, c->d_stage_u8, c->d_src_stage, c->w, c->h);
    c->launches++; c->class_launches[KC_MISC]++;
    CU_TRY(c, cudaMemcpy2DToArrayAsync(dst, 0, 0, c->d_src_stage, trow, trow, c->h, cudaMemcpyDeviceToDevice, c->stream));
    return 0;
}

// per-lane segment tables and chain staging for groups of up to `frames` segments
int ensure_seg_lanes(poppy_cuda_ctx* c, int frames) {
    for (int i = 0; i < c->n_lanes; ++i) {
        auto& l = c->lane[i];
        if (l.seg_cap >= frames) continue;
        cudaFree(l.d_seg); cudaFreeHost(l.h_seg); cudaFree(l.d_seg_stage);
        l.d_seg = nullptr; l.h_seg = nullptr; l.d_seg_stage = nullptr; l.seg_cap = 0;
        CU_TRY(c, dmalloc(&l.d_seg, (size_t)frames));
        CU_TRY(c, cudaMallocHost((void**)&l.h_seg, (size_t)frames * sizeof(SegFrame)));
        CU_TRY(c, dmalloc(&l.d_seg_stage, (size_t)frames * c->pixels()));
        l.seg_cap = frames;
    }
    return 0;
}

// ---- TMA tensor maps (cuTensorMapEncodeTiled through the runtime's driver entry point: no libcuda link dependency) ----
static_assert(sizeof(CUtensorMap) == sizeof(TmaMap) && alignof(CUtensorMap) <= alignof(TmaMap), "TmaMap mirrors CUtensorMap");
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            p = nullptr;
        }
        return (EncodeTiledFn)p;
    }();
    return fn;
}
// planes of 32-bit elements: [n_planes][rows][pitch], box {bx, by, bz}
bool make_plane_map(TmaMap* out, const void* base, int pitch, int rows, size_t plane_stride, size_t n_planes, int bx, int by, int bz) {
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)pitch, (cuuint64_t)rows, (cuuint64_t)n_planes};
    const cuuint64_t strides[2] = {(cuuint64_t)pitch * 4, (cuuint64_t)plane_stride * 4};
    const cuuint32_t box[3] = {(cuuint32_t)bx, (cuuint32_t)by, (cuuint32_t)bz}, es[3] = {1, 1, 1};
    return enc(reinterpret_cast<CUtensorMap*>(out), CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<void*>(base), dims, strides, box, es,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

float* g_level(poppy_cuda_ctx* c, const poppy_cuda_ctx::Lane& l, int k);
float* o_level(poppy_cuda_ctx* c, const poppy_cuda_ctx::Lane& l, int k);

size_t per_frame_scratch_bytes(const poppy_cuda_ctx* c) {
    return c->padded_pixels() * 12 + (c->g_floats + c->o_floats) * 4 + (size_t)c->list_cap * 4 + (size_t)c->n_tiles * 8 +
           (size_t)c->max_tri * (sizeof(int3) + sizeof(TriInverse) + sizeof(TriRaster));
}

int ensure_chunk(poppy_cuda_ctx* c) {
    int want = c->keep_stages ? 1 : c->want_chunk;
    if (want <= 0) {
        // default: keep a lane's scratch under ~12 GiB and give the small pyramid levels enough CTAs
        size_t per = per_frame_scratch_bytes(c);
        want = (int)std::min<size_t>(32, std::max<size_t>(1, (12ull << 30) / std::max<size_t>(per, 1)));
    }
    want = std::max(1, std::min(want, c->max_frames));
    // a second lane only pays when a render spans several chunks
    const int lanes = (c->keep_stages || want >= c->max_frames) ? 1 : kRenderLanes;
    if (c->chunk == want && c->n_lanes == lanes) return 0;
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    for (auto& l : c->lane) if (l.stream) CU_TRY(c, cudaStreamSynchronize(l.stream));
    free_chunk(c);
    const size_t B = want;
    for (int i = 0; i < lanes; ++i) {
        auto& l = c->lane[i];
        CU_TRY(c, dmalloc(&l.d_fp, B));
        CU_TRY(c, dmalloc(&l.d_tri, B * c->max_tri));
        CU_TRY(c, dmalloc(&l.d_inv, B * c->max_tri));
        CU_TRY(c, dmalloc(&l.d_rast, B * c->max_tri));
        CU_TRY(c, dmalloc(&l.d_trimap, c->keep_stages ? c->pixels() : 1));
        CU_TRY(c, dmalloc(&l.d_tile_cnt, B * c->n_tiles));
        CU_TRY(c, dmalloc(&l.d_tile_off, B * (c->n_tiles + 1)));
        CU_TRY(c, dmalloc(&l.d_tile_list, B * c->list_cap));
        CU_TRY(c, dmalloc(&l.d_overflow, B));
        CU_TRY(c, dmalloc(&l.d_warped, B * 2 * c->padded_pixels()));
        CU_TRY(c, dmalloc(&l.d_mask0, B * c->padded_pixels()));
        CU_TRY(c, dmalloc(&l.d_g, B * c->g_floats));
        CU_TRY(c, dmalloc(&l.d_o, B * c->o_floats));
        CU_TRY(c, dmalloc(&l.d_excess, B * 3 * c->mm_stride));
        CU_TRY(c, dmalloc(&l.d_block_dev, 2 * B * (size_t)div_up(c->w, CALM_BLOCK_W) * div_up(c->h, CALM_BLOCK_H)));
        CU_TRY(c, dmalloc(&l.d_block_flags, B * (size_t)div_up(c->w, CALM_BLOCK_W) * div_up(c->h, CALM_BLOCK_H)));
        CU_TRY(c, dmalloc(&l.d_chunk_flags, B * (size_t)div_up(c->w, UNSHARP_STRIP_W) * div_up(c->h, kSparseChunkRows)));
        CU_TRY(c, dmalloc(&l.d_tile_flags, B * (size_t)div_up(c->w, 128) * div_up(c->h, 32)));
        CU_TRY(c, dmalloc(&l.d_calm_counts, B));
        CU_TRY(c, cudaMallocHost((void**)&l.h_calm_counts, B * sizeof(int)));
        CU_TRY(c, cudaMallocHost((void**)&l.h_fp, B * sizeof(FrameParams)));
        CU_TRY(c, cudaMallocHost((void**)&l.h_tri, std::max<size_t>(B * c->max_tri, 1) * 3 * sizeof(int32_t)));
    }
    c->chunk = want;
    c->n_lanes = lanes;
    {   // level table of k_pyramid_tail: the offsets depend on the chunk size
        std::vector<TailLevel> tl(c->levels + 1);
        for (int k = 0; k <= c->levels; ++k)
            tl[k] = TailLevel{c->lv[k].w, c->lv[k].h, c->lv[k].pitch, 0, c->lv[k].plane_stride, c->g_off[k] * (size_t)want, c->o_off[k] * (size_t)want};
        cudaFree(c->d_tail_levels);
        c->d_tail_levels = nullptr;
        CU_TRY(c, dmalloc(&c->d_tail_levels, tl.size()));
        CU_TRY(c, cudaMemcpy(c->d_tail_levels, tl.data(), tl.size() * sizeof(TailLevel), cudaMemcpyHostToDevice));
    }
    // tensor maps of every level's collapse (level k fine, level k+1 coarse). A level too small for the boxes keeps an
    // all-zero entry and runs k_collapse_roll: it has no interior tile.
    for (int i = 0; i < lanes; ++i) {
        auto& l = c->lane[i];
        l.maps.assign(c->levels, CollapseMaps());
        for (int k = 0; k < c->levels; ++k) {
            const LevelDesc &fl = c->lv[k], &cl = c->lv[k + 1];
            CollapseMaps& m = l.maps[k];
            bool ok;
            if (k == 0) {
                ok = make_plane_map(&m.fine, l.d_warped, c->pitch0(), c->h, c->padded_pixels(), 2 * B, 128, 2, 2) &&
                     make_plane_map(&m.mask, l.d_mask0, c->pitch0(), c->h, c->padded_pixels(), B, 128, 2, 1);
            } else {
                // keep the 128 x 2 box inside the tensor
                if (fl.pitch < 128 || fl.h < 2) continue;
                ok = make_plane_map(&m.fine, g_level(c, l, k), fl.pitch, fl.h, fl.plane_stride, 7 * B, 128, 2, 7);
                m.mask = m.fine;
            }
            if (ok && cl.pitch < 72) { m = CollapseMaps(); continue; }
            ok = ok && make_plane_map(&m.gc, g_level(c, l, k + 1), cl.pitch, cl.h, cl.plane_stride, 7 * B, 72, 1, 6) &&
                 make_plane_map(&m.oc, o_level(c, l, k + 1), cl.pitch, cl.h, cl.plane_stride, 3 * B, 72, 1, 3);
            if (!ok) {
                free_chunk(c);       // the next render retries instead of running without the maps
                return fail(c, POPPY_CUDA_ERR_CUDA, "cuTensorMapEncodeTiled %s for the collapse of level %d",
                            tensor_map_encoder() ? "failed" : "is not available from the driver", k);
            }
        }
    }
    return 0;
}

// level k block of a chunk: all frames' planes of that level are contiguous
float* g_level(poppy_cuda_ctx* c, const poppy_cuda_ctx::Lane& l, int k) { return l.d_g + c->g_off[k] * c->chunk; }
float* o_level(poppy_cuda_ctx* c, const poppy_cuda_ctx::Lane& l, int k) { return l.d_o + c->o_off[k] * c->chunk; }

// tensor maps of level k's collapse, or null where the level has none (all-zero map = not built)
const CollapseMaps* level_maps(const poppy_cuda_ctx::Lane& l, int k) {
    if (k >= (int)l.maps.size()) return nullptr;
    const CollapseMaps& m = l.maps[k];
    bool any = false;
    for (unsigned long long v : m.gc.v) any = any || v != 0;
    return any ? &m : nullptr;
}

cudaEvent_t get_event(poppy_cuda_ctx* c) {
    if (!c->event_pool.empty()) { cudaEvent_t e = c->event_pool.back(); c->event_pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

struct Scope {   // counts a launch and, when stage timing is on, brackets it with events
    poppy_cuda_ctx* c; int cls; cudaStream_t st; TimedLaunch t{};
    Scope(poppy_cuda_ctx* c_, int cls_, cudaStream_t st_) : c(c_), cls(cls_), st(st_) {
        c->launches++;
        c->class_launches[cls]++;
        if (c->stage_timing) { t.cls = cls; t.a = get_event(c); t.b = get_event(c); cudaEventRecord(t.a, st); }
    }
    ~Scope() {
        if (c->stage_timing) { cudaEventRecord(t.b, st); c->timed.push_back(t); }
    }
};

void collect_timing(poppy_cuda_ctx* c) {
    for (auto& t : c->timed) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) c->class_ms[t.cls] += ms;
        c->event_pool.push_back(t.a);
        c->event_pool.push_back(t.b);
    }
    c->timed.clear();
}

// fold the flagged-chunk counts of finished calm-route chunks into the running share (never blocks unless `wait`)
void harvest_calm_stats(poppy_cuda_ctx* c, bool wait) {
    const int chunks_per_frame = div_up(c->w, UNSHARP_STRIP_W) * div_up(c->h, kSparseChunkRows);
    for (auto& l : c->lane) {
        if (!l.calm_pending) continue;
        if (wait) cudaEventSynchronize(l.ev_calm);
        else if (cudaEventQuery(l.ev_calm) != cudaSuccess) { cudaGetLastError(); continue; }
        long long flagged = 0;
        for (int i = 0; i < l.calm_pending; ++i) flagged += l.h_calm_counts[i];
        const double share = (double)flagged / ((double)l.calm_pending * chunks_per_frame);
        c->calm_share = 0.5 * c->calm_share + 0.5 * share;
        // content that keeps flagging most chunks is probed less and less often; anything calmer resets the interval
        c->probe_every = share > 0.5 ? std::min(c->probe_every * 2, 64u) : kCalmProbeEvery;
        l.calm_pending = 0;
    }
}

// One step of a group of segments (poppy_cuda_render_segments): frame i of the chunk is step `step` of segment s0 + i, its
// shape / mask ratio is entry `row` of the call's arrays and its triangle list entry row * n_seg + s0 + i.
struct SegChunk { int s0, step, row; };

// tri_idx == nullptr: the triangles come from the resident plan, tri_off pointing into its offsets (frame `first` of this call
// is plan frame plan_first + first)
int render_chunk(poppy_cuda_ctx* c, int slot0, int first, int nb, const float* shape, const double* mask, const int32_t* tri_idx,
                 const int32_t* tri_off, bool chain, poppy_cuda_ctx::Lane& ln, const SegChunk* sg = nullptr) {
    cudaStream_t st = ln.stream;
    CU_TRY(c, cudaEventSynchronize(ln.ev_staged));       // the lane's staging buffers are free again
    FrameParams* hp = ln.h_fp;
    int32_t* ht = ln.h_tri;
    int tri_total = 0, tri_max = 0, seg_n_max = 0;
    const int K = (int)c->seg.size(), W = c->seg_window;
    for (int i = 0; i < nb; ++i) {
        const int f = sg ? sg->row * K + sg->s0 + i : first + i;       // triangle list entry
        const int r = sg ? sg->row : f;                                 // ratio entry
        const int nt = tri_off[f + 1] - tri_off[f];
        if (nt < 0 || nt > c->max_tri) return fail(c, POPPY_CUDA_ERR_CAPACITY, "frame %d has %d triangles (max %d)", f, nt, c->max_tri);
        if (tri_idx && nt)         // validated by poppy_cuda_render_range
            std::memcpy(ht + (size_t)tri_total * 3, tri_idx + (size_t)tri_off[f] * 3, (size_t)nt * 3 * sizeof(int32_t));
        FrameParams& p = hp[i];
        p.shape = shape[r];
        p.one_minus_r = (float)(1.0 - (double)p.shape);
        p.mask_alpha = 1.0 - mask[r];
        p.mask_beta = -mask[r];
        p.amount = (float)(1.0 - std::sin(mask[r] * M_PI));
        p.n_tri = nt;
        p.tri_base = tri_total;
        p.dst_slot = sg ? (sg->s0 + i) * W + sg->step % W : slot0 + f;
        tri_total += nt;
        tri_max = std::max(tri_max, nt);
        if (sg) {
            const poppy_cuda_ctx::Segment& S = c->seg[sg->s0 + i];
            SegFrame& q = ln.h_seg[i];
            q.src1 = sg->step == 0 ? S.t[0] : S.t[2];
            q.src2 = S.t[1];
            q.basis = c->d_seg_basis + (size_t)(sg->s0 + i) * c->padded_pixels();
            q.pts2 = c->d_seg_pts2 + (size_t)(sg->s0 + i) * c->max_points;
            q.n_points = S.n;
            q.pad = 0;
            seg_n_max = std::max(seg_n_max, S.n);
        }
    }
    CU_TRY(c, cudaMemcpyAsync(ln.d_fp, hp, nb * sizeof(FrameParams), cudaMemcpyHostToDevice, st));
    if (sg) CU_TRY(c, cudaMemcpyAsync(ln.d_seg, ln.h_seg, nb * sizeof(SegFrame), cudaMemcpyHostToDevice, st));
    if (tri_idx && tri_total)
        CU_TRY(c, cudaMemcpyAsync(ln.d_tri, ht, (size_t)tri_total * 3 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CU_TRY(c, cudaEventRecord(ln.ev_staged, st));
    // the chunk's packed triangles: the lane's staging copy, or their place in the resident plan (same packing)
    const int3* chunk_tri = tri_idx ? ln.d_tri : c->d_plan_tri + tri_off[first];

    // a chain continues from the frame before it: the previous frame of this call, or - when a chain is rendered slice by
    // slice - the last frame of the previous call (ring slot slot0 + first - 1, whose pixels are still in t_src[2])
    const bool chained = chain && (slot0 + first) > 0;
    const float2* p1 = chained ? c->d_morphed + (size_t)(slot0 + first - 1) * c->max_points : c->d_pts1;
    const cudaTextureObject_t src1 = chained ? c->t_src[2] : c->t_src[0];
    float2* morphed = c->d_morphed + (size_t)(slot0 + first) * c->max_points;
    const int n = c->n_points, w = c->w, h = c->h, L = c->levels;

    // segments: the chunk's frames are consecutive segments, so their previous steps' points and their outputs lie a
    // constant W * max_points apart in the ring, their step-0 points max_points apart
    const size_t ring_stride = (size_t)W * c->max_points;
    const float2* sp1 = !sg ? nullptr
                      : sg->step == 0 ? c->d_seg_pts1 + (size_t)sg->s0 * c->max_points
                                      : c->d_morphed + ((size_t)sg->s0 * W + (sg->step - 1) % W) * c->max_points;
    const size_t sp1_stride = sg && sg->step == 0 ? (size_t)c->max_points : ring_stride;
    float2* smorphed = sg ? c->d_morphed + ((size_t)sg->s0 * W + sg->step % W) * c->max_points : nullptr;

    {   Scope s(c, KC_POINTS, st);
        if (sg) launch_lerp_points_seg(st, sp1, sp1_stride, ln.d_seg, ln.d_fp, smorphed, ring_stride, seg_n_max, nb, w, h);
        else launch_lerp_points(st, p1, 0, c->d_pts2, ln.d_fp, morphed, c->max_points, n, nb, w, h);
    }
    CU_TRY(c, cudaMemsetAsync(ln.d_tile_cnt, 0, (size_t)nb * c->n_tiles * sizeof(int), st));
    {   Scope s(c, KC_GEOMETRY, st);
        if (sg)
            launch_tri_geometry_seg(st, chunk_tri, ln.d_fp, sp1, sp1_stride, ln.d_seg, smorphed, ring_stride, c->max_tri, tri_max, nb,
                                    w, h, ln.d_inv, ln.d_rast, ln.d_tile_cnt);
        else
            launch_tri_geometry(st, chunk_tri, ln.d_fp, p1, 0, c->d_pts2, morphed, c->max_points, c->max_tri, tri_max, nb, w, h,
                                ln.d_inv, ln.d_rast, ln.d_tile_cnt);
    }
    {   Scope s(c, KC_BIN, st);
        c->launches++;          // scan + fill
        launch_bin_triangles(st, ln.d_rast, ln.d_fp, c->max_tri, tri_max, nb, w, h, ln.d_tile_cnt, ln.d_tile_off,
                             ln.d_overflow, ln.d_tile_list, c->list_cap);
    }
    {   Scope s(c, KC_WARP, st);
        if (sg)
            launch_raster_warp_seg(st, ln.d_rast, ln.d_inv, ln.d_fp, c->max_tri, ln.d_tile_off, ln.d_tile_list, c->list_cap,
                                   ln.d_overflow, ln.d_seg, ln.d_warped, c->pitch0(), c->padded_pixels(), w, h, nb);
        else
            launch_raster_warp(st, ln.d_rast, ln.d_inv, ln.d_fp, c->max_tri, ln.d_tile_off, ln.d_tile_list, c->list_cap,
                               ln.d_overflow, src1, c->t_src[1], ln.d_warped, c->pitch0(), c->padded_pixels(),
                               c->keep_stages ? ln.d_trimap : nullptr, w, h, nb);
    }
    {   Scope s(c, KC_PYR_DOWN, st);
        if (sg)
            launch_pyr_down0_seg(st, ln.d_warped, c->pitch0(), c->padded_pixels(), ln.d_seg, c->pitch0(), ln.d_fp, w, h, ln.d_mask0,
                                 c->padded_pixels(), g_level(c, ln, 1), c->lv[1], nb);
        else
            launch_pyr_down0(st, ln.d_warped, c->pitch0(), c->padded_pixels(), c->d_mbasis, c->pitch0(), ln.d_fp, w, h, ln.d_mask0,
                             c->padded_pixels(), g_level(c, ln, 1), c->lv[1], nb);
    }
    const int k0 = c->tail_k0;                  // levels k0 .. L: one launch
    for (int k = 1; k < (k0 ? k0 : L); ++k) {
        Scope s(c, KC_PYR_DOWN, st);
        launch_pyr_down(st, g_level(c, ln, k), c->lv[k], g_level(c, ln, k + 1), c->lv[k + 1], nb);
    }
    if (k0) {
        Scope s(c, KC_COLLAPSE, st);
        launch_pyramid_tail(st, ln.d_g, ln.d_o, c->d_tail_levels, k0, L, nb);
    } else {
        Scope s(c, KC_COLLAPSE, st);
        launch_blend_coarsest(st, g_level(c, ln, L), c->lv[L], o_level(c, ln, L), nb);
    }
    for (int k = (k0 ? k0 : L) - 1; k >= 1; --k) {
        Scope s(c, KC_COLLAPSE, st);
        launch_collapse(st, g_level(c, ln, k), c->lv[k], g_level(c, ln, k + 1), o_level(c, ln, k + 1), c->lv[k + 1], o_level(c, ln, k), nb,
                        level_maps(ln, k));
    }
    // ---- level 0: collapse + unsharp_mask + 8-bit store, by one of two bit-identical routes ---------------------------
    const int chunks_per_frame = div_up(w, UNSHARP_STRIP_W) * div_up(h, kSparseChunkRows);
    harvest_calm_stats(c, false);
    bool calm_route;
    if (c->keep_stages || c->unsharp_mode == 1) calm_route = false;
    else if (c->unsharp_mode == 2) calm_route = true;
    else calm_route = c->calm_share <= kCalmRouteMaxShare;
    if (calm_route) {
        {   Scope s(c, KC_COLLAPSE, st);
            launch_collapse0_emit(st, ln.d_warped, c->pitch0(), c->padded_pixels(), ln.d_mask0, c->pitch0(), c->padded_pixels(), w, h,
                                  g_level(c, ln, 1), o_level(c, ln, 1), c->lv[1], ln.d_fp, c->d_frames, c->frame_bytes(), ln.d_excess,
                                  c->mm_pitch, c->mm_stride, nb, level_maps(ln, 0));
        }
        {   Scope s(c, KC_CALM, st);
            c->launches += 2;       // byte scan + block flags + chunk flags
            launch_calm_analysis(st, c->d_frames, c->frame_bytes(), ln.d_fp, ln.d_excess, c->mm_pitch, c->mm_stride, w, h, nb,
                                 kSparseChunkRows, ln.d_block_dev, ln.d_block_flags, ln.d_chunk_flags, ln.d_tile_flags, ln.d_calm_counts,
                                 c->d_calm_total, 0);
            c->calm_chunks_total += (uint64_t)nb * chunks_per_frame;
        }
        if (ln.calm_pending) { CU_TRY(c, cudaEventSynchronize(ln.ev_calm)); harvest_calm_stats(c, false); }
        CU_TRY(c, cudaMemcpyAsync(ln.h_calm_counts, ln.d_calm_counts, (size_t)nb * sizeof(int), cudaMemcpyDeviceToHost, st));
        CU_TRY(c, cudaEventRecord(ln.ev_calm, st));
        ln.calm_pending = nb;
        {   Scope s(c, KC_COLLAPSE, st);
            launch_collapse0(st, ln.d_warped, c->pitch0(), c->padded_pixels(), ln.d_mask0, c->pitch0(), c->padded_pixels(), w, h,
                             g_level(c, ln, 1), o_level(c, ln, 1), c->lv[1], o_level(c, ln, 0), c->lv[0], nb, ln.d_tile_flags, level_maps(ln, 0));
        }
        {   Scope s(c, KC_UNSHARP, st);
            launch_unsharp_store(st, o_level(c, ln, 0), c->lv[0], ln.d_fp, c->d_frames, c->frame_bytes(), nb, kSparseChunkRows,
                                 ln.d_chunk_flags);
        }
    } else {
        // dense route: the level-0 collapse of the whole chunk to float planes, then the exact unsharp pass on every pixel
        {   Scope s(c, KC_COLLAPSE, st);
            launch_collapse0(st, ln.d_warped, c->pitch0(), c->padded_pixels(), ln.d_mask0, c->pitch0(), c->padded_pixels(), w, h,
                             g_level(c, ln, 1), o_level(c, ln, 1), c->lv[1], o_level(c, ln, 0), c->lv[0], nb, nullptr, level_maps(ln, 0));
        }
        {   Scope s(c, KC_UNSHARP, st);
            launch_unsharp_store(st, o_level(c, ln, 0), c->lv[0], ln.d_fp, c->d_frames, c->frame_bytes(), nb, 0, nullptr);
        }
        c->dense_chunks_total += (uint64_t)nb * chunks_per_frame;
        if (c->unsharp_mode == 0 && !c->keep_stages && (++c->route_tick % c->probe_every) == 0 && !ln.calm_pending) {
            // statistic only: the byte scan of the finished frames (no clamp-excess information on this route)
            Scope s(c, KC_CALM, st);
            c->launches += 2;
            CU_TRY(c, cudaMemsetAsync(ln.d_excess, 0, (size_t)nb * 3 * c->mm_stride, st));
            launch_calm_analysis(st, c->d_frames, c->frame_bytes(), ln.d_fp, ln.d_excess, c->mm_pitch, c->mm_stride, w, h, nb,
                                 kSparseChunkRows, ln.d_block_dev, ln.d_block_flags, ln.d_chunk_flags, ln.d_tile_flags, ln.d_calm_counts,
                                 c->d_probe_total, 0);
            CU_TRY(c, cudaMemcpyAsync(ln.h_calm_counts, ln.d_calm_counts, (size_t)nb * sizeof(int), cudaMemcpyDeviceToHost, st));
            CU_TRY(c, cudaEventRecord(ln.ev_calm, st));
            ln.calm_pending = nb;
        }
    }
    if (sg) {
        // every segment's chain source becomes this step's frame: one conversion for the chunk, one array copy per segment
        Scope s(c, KC_MISC, st);
        launch_bgr_to_bgrx_frames(st, c->d_frames, c->frame_bytes(), ln.d_fp, ln.d_seg_stage, w, h, nb);
        for (int i = 0; i < nb; ++i)
            CU_TRY(c, cudaMemcpy2DToArrayAsync(c->seg[sg->s0 + i].a[2], 0, 0, ln.d_seg_stage + (size_t)i * c->pixels(), (size_t)w * 4,
                                               (size_t)w * 4, h, cudaMemcpyDeviceToDevice, st));
    } else if (chain) {
        Scope s(c, KC_MISC, st);
        launch_bgr_to_bgrx(st, c->d_frames + (size_t)(slot0 + first + nb - 1) * c->frame_bytes(), c->d_src_stage, w, h);
        CU_TRY(c, cudaMemcpy2DToArrayAsync(c->a_src[2], 0, 0, c->d_src_stage, (size_t)w * 4, (size_t)w * 4, h,
                                           cudaMemcpyDeviceToDevice, st));
    }
    CU_TRY(c, cudaGetLastError());
    return 0;
}

}  // namespace

// =================================================================================================================
extern "C" {

const char* poppy_cuda_version(void) { return "poppy_cuda 0.1 sm_100a"; }

int poppy_cuda_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char* poppy_cuda_last_error(const poppy_cuda_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int poppy_cuda_create(poppy_cuda_ctx** out, int device, int width, int height, int pyramid_levels, int max_points,
                      int max_triangles, int max_batch_frames) {
    if (!out) return fail(nullptr, POPPY_CUDA_ERR_INVALID, "out is null");
    *out = nullptr;
    if (width <= 0 || height <= 0 || width >= 32767 || height >= 32767)
        return fail(nullptr, POPPY_CUDA_ERR_INVALID, "frame size %dx%d out of range (cv::remap needs < 32767)", width, height);
    if (pyramid_levels < 1 || max_points < 1 || max_triangles < 1 || max_batch_frames < 1)
        return fail(nullptr, POPPY_CUDA_ERR_INVALID, "pyramid_levels/max_points/max_triangles/max_batch_frames out of range");
    int ndev = poppy_cuda_device_count();
    if (ndev <= 0) return fail(nullptr, POPPY_CUDA_ERR_NO_DEVICE, "no CUDA device: the morph renderer has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(nullptr, POPPY_CUDA_ERR_INVALID, "device %d not in [0,%d)", device, ndev);
    poppy_cuda_ctx* c = new poppy_cuda_ctx();
    c->device = device; c->w = width; c->h = height; c->levels = pyramid_levels;
    c->max_points = max_points; c->max_tri = max_triangles; c->max_frames = max_batch_frames;
    auto bail = [&](int rc) { g_create_error = c->err; poppy_cuda_destroy(c); return rc; };
#define CR_TRY(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) { \
        fail(c, POPPY_CUDA_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e_)); return bail(POPPY_CUDA_ERR_CUDA); } } while (0)
    CR_TRY(cudaSetDevice(device));
    CR_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CR_TRY(cudaEventCreate(&c->ev_begin));
    CR_TRY(cudaEventCreate(&c->ev_end));
    CR_TRY(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    CR_TRY(cudaEventCreateWithFlags(&c->ev_rendered, cudaEventDisableTiming));
    CR_TRY(cudaEventCreateWithFlags(&c->ev_copied, cudaEventDisableTiming));
    for (auto& l : c->lane) {
        CR_TRY(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
        CR_TRY(cudaEventCreateWithFlags(&l.ev_staged, cudaEventDisableTiming));
        CR_TRY(cudaEventCreateWithFlags(&l.ev_done, cudaEventDisableTiming));
        CR_TRY(cudaEventCreateWithFlags(&l.ev_calm, cudaEventDisableTiming));
    }
    // pyramid geometry: (n+1)/2 per level, 1x1 levels repeat (cv::pyrDown, pyramids.cpp:1260-1303)
    c->lv.resize(pyramid_levels + 1);
    c->g_off.assign(pyramid_levels + 2, 0);
    c->o_off.assign(pyramid_levels + 2, 0);
    int lw = width, lh = height;
    for (int k = 0; k <= pyramid_levels; ++k) {
        LevelDesc& d = c->lv[k];
        d.w = lw; d.h = lh; d.pitch = (lw + 31) & ~31; d.plane_stride = (size_t)d.pitch * lh;
        c->g_off[k] = c->g_floats;
        c->o_off[k] = c->o_floats;
        if (k >= 1) c->g_floats += 7 * d.plane_stride;
        c->o_floats += 3 * d.plane_stride;
        lw = (lw + 1) / 2; lh = (lh + 1) / 2;
    }
    // the pyramid's tail: from the first level no larger than 32 x 32 on, all levels run in one launch
    for (int k = 1; k < pyramid_levels; ++k)
        if (c->lv[k].w <= 32 && c->lv[k].h <= 32) { c->tail_k0 = k; break; }
    // triangle binning: 64x32 screen tiles; list capacity per frame (a frame that needs more falls back to testing
    // every triangle in every tile, see k_raster_warp)
    {
        const long long tiles = (long long)((width + RW_TW - 1) / RW_TW) * ((height + RW_TH - 1) / RW_TH);
        c->n_tiles = (int)tiles;
        const long long all = tiles * max_triangles;
        const long long want = std::max<long long>(8LL * max_triangles + 4 * tiles, 1LL << 20);
        c->list_cap = (int)std::min<long long>(all, want);
    }
    c->mm_pitch = (div_up(width, CALM_BLOCK_W) + 15) & ~15;
    c->mm_stride = (size_t)c->mm_pitch * div_up(height, CALM_BLOCK_H);
    CR_TRY(dmalloc(&c->d_probe_total, (size_t)1));
    CR_TRY(dmalloc(&c->d_calm_total, (size_t)1));
    CR_TRY(cudaMemset(c->d_calm_total, 0, sizeof(unsigned long long)));
    const size_t px = c->pixels();
    CR_TRY(dmalloc(&c->d_src_stage, px));
    for (int i = 0; i < 3; ++i) {
        const cudaChannelFormatDesc fmt = cudaCreateChannelDesc<uchar4>();
        CR_TRY(cudaMallocArray(&c->a_src[i], &fmt, (size_t)width, (size_t)height, cudaArrayTextureGather));
        cudaResourceDesc res{};
        res.resType = cudaResourceTypeArray;
        res.res.array.array = c->a_src[i];
        cudaTextureDesc td{};
        td.addressMode[0] = td.addressMode[1] = cudaAddressModeBorder;      // BORDER_CONSTANT(0)
        td.filterMode = cudaFilterModePoint;
        td.readMode = cudaReadModeElementType;
        td.normalizedCoords = 0;
        CR_TRY(cudaCreateTextureObject(&c->t_src[i], &res, &td, nullptr));
    }
    CR_TRY(dmalloc(&c->d_mbasis, c->padded_pixels()));
    CR_TRY(dmalloc(&c->d_pts1_raw, (size_t)max_points));
    CR_TRY(dmalloc(&c->d_pts2_raw, (size_t)max_points));
    CR_TRY(dmalloc(&c->d_pts1, (size_t)max_points));
    CR_TRY(dmalloc(&c->d_pts2, (size_t)max_points));
    CR_TRY(dmalloc(&c->d_morphed, (size_t)max_points * max_batch_frames));
    CR_TRY(dmalloc(&c->d_frames, c->frame_bytes() * max_batch_frames));
    CR_TRY(dmalloc(&c->d_sum, (size_t)1));
#undef CR_TRY
    *out = c;
    return 0;
}

void poppy_cuda_destroy(poppy_cuda_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    for (auto& l : c->lane) if (l.stream) cudaStreamSynchronize(l.stream);
    collect_timing(c);
    for (cudaEvent_t e : c->event_pool) cudaEventDestroy(e);
    for (cudaEvent_t e : c->tickets) if (e) cudaEventDestroy(e);
    free_chunk(c);
    free_segments(c);
    cudaFree(c->d_src_stage); cudaFree(c->d_mbasis); cudaFree(c->d_stage_u8); cudaFree(c->d_stage_f32);
    for (int i = 0; i < 3; ++i) {
        if (c->t_src[i]) cudaDestroyTextureObject(c->t_src[i]);
        if (c->a_src[i]) cudaFreeArray(c->a_src[i]);
    }
    cudaFree(c->d_pts1_raw); cudaFree(c->d_pts2_raw); cudaFree(c->d_pts1); cudaFree(c->d_pts2); cudaFree(c->d_morphed);
    cudaFree(c->d_tail_levels);
    cudaFree(c->ffv1.d_sym); cudaFree(c->ffv1.d_slots); cudaFree(c->ffv1.d_packets); cudaFree(c->ffv1.d_tables);
    cudaFree(c->ffv1.d_scratch); cudaFree(c->ffv1.d_sizes); cudaFree(c->ffv1.d_frame_sizes); cudaFree(c->ffv1.d_offsets);
    cudaFree(c->ffv1.d_slot_of); cudaFree(c->ffv1.d_overflow);
    if (c->ffv1.h_overflow) cudaFreeHost(c->ffv1.h_overflow);
    cudaFree(c->d_frames); cudaFree(c->d_i420); cudaFree(c->d_sum); cudaFree(c->d_calm_total); cudaFree(c->d_probe_total); cudaFree(c->d_plan_tri);
    if (c->ev_begin) cudaEventDestroy(c->ev_begin);
    if (c->ev_end) cudaEventDestroy(c->ev_end);
    if (c->ev_rendered) cudaEventDestroy(c->ev_rendered);
    if (c->ev_copied) cudaEventDestroy(c->ev_copied);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    for (auto& l : c->lane) {
        if (l.ev_staged) cudaEventDestroy(l.ev_staged);
        if (l.ev_done) cudaEventDestroy(l.ev_done);
        if (l.ev_calm) cudaEventDestroy(l.ev_calm);
        if (l.stream) cudaStreamDestroy(l.stream);
    }
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int poppy_cuda_get_info(const poppy_cuda_ctx* c, int* width, int* height, int* pyramid_levels, int* max_points,
                        int* max_triangles, int* max_batch_frames) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (width) *width = c->w;
    if (height) *height = c->h;
    if (pyramid_levels) *pyramid_levels = c->levels;
    if (max_points) *max_points = c->max_points;
    if (max_triangles) *max_triangles = c->max_tri;
    if (max_batch_frames) *max_batch_frames = c->max_frames;
    return 0;
}

int poppy_cuda_set_keep_stages(poppy_cuda_ctx* c, int keep) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    c->keep_stages = keep != 0;
    return 0;
}

int poppy_cuda_set_chunk_frames(poppy_cuda_ctx* c, int frames) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (frames < 1) return fail(c, POPPY_CUDA_ERR_INVALID, "chunk frames must be >= 1");
    c->want_chunk = frames;
    return 0;
}

int poppy_cuda_set_tile_list_capacity(poppy_cuda_ctx* c, int entries) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (entries < 1) return fail(c, POPPY_CUDA_ERR_INVALID, "tile list capacity must be >= 1");
    CU_TRY(c, cudaSetDevice(c->device));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    c->list_cap = entries;
    free_chunk(c);            // reallocated with the new capacity by the next render
    return 0;
}

int poppy_cuda_set_unsharp_mode(poppy_cuda_ctx* c, int mode) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (mode < 0 || mode > 2) return fail(c, POPPY_CUDA_ERR_INVALID, "unsharp mode must be 0 (adaptive), 1 (dense) or 2 (calm route)");
    c->unsharp_mode = mode;
    return 0;
}

int poppy_cuda_unsharp_stats(poppy_cuda_ctx* c, uint64_t* chunks_exact, uint64_t* chunks_total) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    CU_TRY(c, cudaSetDevice(c->device));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    for (auto& l : c->lane) if (l.stream) CU_TRY(c, cudaStreamSynchronize(l.stream));
    harvest_calm_stats(c, true);
    unsigned long long v = 0;
    CU_TRY(c, cudaMemcpy(&v, c->d_calm_total, sizeof v, cudaMemcpyDeviceToHost));
    CU_TRY(c, cudaMemset(c->d_calm_total, 0, sizeof v));
    if (chunks_exact) *chunks_exact = v + c->dense_chunks_total;
    if (chunks_total) *chunks_total = c->calm_chunks_total + c->dense_chunks_total;
    c->calm_chunks_total = c->dense_chunks_total = 0;
    return 0;
}

int poppy_cuda_set_stage_timing(poppy_cuda_ctx* c, int enable) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    c->stage_timing = enable != 0;
    return 0;
}

// upload staging of the pair, allocated on first use and kept (no cudaMalloc / cudaFree per call): 8-bit for the images,
// float (99.5 MB at 4K) only once a caller supplies gabor2 itself
static int ensure_pair_staging(poppy_cuda_ctx* c, int which) {
    if (which != 2 && !c->d_stage_u8) CU_TRY(c, dmalloc(&c->d_stage_u8, c->frame_bytes()));
    if (which == 2 && !c->d_stage_f32) CU_TRY(c, dmalloc(&c->d_stage_f32, c->pixels() * 3));
    return 0;
}

int poppy_cuda_set_image(poppy_cuda_ctx* c, int which, const void* data, size_t step) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (!data || which < 0 || which > 3) return fail(c, POPPY_CUDA_ERR_INVALID, "bad image selector or null pointer");
    const size_t row = (size_t)c->w * 3, grow = row * sizeof(float), trow = (size_t)c->w * 4;
    if (step < (which == 2 ? grow : row)) return fail(c, POPPY_CUDA_ERR_INVALID, "row stride smaller than a row");
    CU_TRY(c, cudaSetDevice(c->device));
    if (int rc = ensure_pair_staging(c, which)) return rc;
    if (which != 2) {
        CU_TRY(c, cudaMemcpy2DAsync(c->d_stage_u8, row, data, step, row, c->h, cudaMemcpyHostToDevice, c->stream));
        launch_bgr_to_bgrx(c->stream, c->d_stage_u8, c->d_src_stage, c->w, c->h);
        CU_TRY(c, cudaMemcpy2DToArrayAsync(c->a_src[which == 0 ? 0 : 1], 0, 0, c->d_src_stage, trow, trow, c->h,
                                           cudaMemcpyDeviceToDevice, c->stream));
    } else {
        CU_TRY(c, cudaMemcpy2DAsync(c->d_stage_f32, grow, data, step, grow, c->h, cudaMemcpyHostToDevice, c->stream));
        launch_mask_basis(c->stream, c->d_stage_f32, c->d_mbasis, c->pitch0(), c->w, c->h);
    }
    c->launches++; c->class_launches[KC_MISC]++;
    CU_TRY(c, cudaGetLastError());
    if (which == 3) {
        // corrected2 is still in the 8-bit staging (same stream): the mask basis from it, gabor2 never stored
        Scope s(c, KC_MISC, c->stream);
        CU_TRY(c, launch_gabor_mask_basis(c->stream, c->d_stage_u8, c->d_mbasis, c->pitch0(), c->w, c->h));
        c->have_image[1] = true;
    }
    c->have_image[which == 3 ? 2 : which] = true;
    c->have_pair = c->have_image[0] && c->have_image[1] && c->have_image[2];
    return 0;
}

int poppy_cuda_set_pair(poppy_cuda_ctx* c, const uint8_t* bgr1, size_t step1, const uint8_t* bgr2, size_t step2,
                        const float* gabor, size_t gstep) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (!bgr1 || !bgr2) return fail(c, POPPY_CUDA_ERR_INVALID, "null image pointer");
    int rc;
    if ((rc = poppy_cuda_set_image(c, 0, bgr1, step1)) != 0) return rc;
    if (!gabor) rc = poppy_cuda_set_image(c, 3, bgr2, step2);      // no gabor2: derive the mask basis from corrected2
    else if ((rc = poppy_cuda_set_image(c, 1, bgr2, step2)) == 0) rc = poppy_cuda_set_image(c, 2, gabor, gstep);
    if (rc != 0) return rc;
    // the host arrays may be pinned (a truly asynchronous copy) and reused by the caller right after this call
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int poppy_cuda_set_source1_from_slot(poppy_cuda_ctx* c, int slot) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (slot < 0 || slot >= c->max_frames) return fail(c, POPPY_CUDA_ERR_INVALID, "bad frame slot");
    CU_TRY(c, cudaSetDevice(c->device));
    const size_t trow = (size_t)c->w * 4;
    launch_bgr_to_bgrx(c->stream, c->d_frames + (size_t)slot * c->frame_bytes(), c->d_src_stage, c->w, c->h);
    CU_TRY(c, cudaMemcpy2DToArrayAsync(c->a_src[0], 0, 0, c->d_src_stage, trow, trow, c->h, cudaMemcpyDeviceToDevice, c->stream));
    c->launches++; c->class_launches[KC_MISC]++;
    CU_TRY(c, cudaGetLastError());
    c->have_image[0] = true;
    c->have_pair = c->have_image[0] && c->have_image[1] && c->have_image[2];
    return 0;
}

int poppy_cuda_set_points(poppy_cuda_ctx* c, const float* pts1, const float* pts2, int n) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    // fewer than 3 points give no triangle: like the reference (an empty Delaunay mesh) the frame is then the blend of the
    // unwarped pair
    if ((n > 0 && (!pts1 || !pts2)) || n < 0) return fail(c, POPPY_CUDA_ERR_INVALID, "bad point sets");
    if (n > c->max_points) return fail(c, POPPY_CUDA_ERR_CAPACITY, "%d points (max %d)", n, c->max_points);
    CU_TRY(c, cudaSetDevice(c->device));
    if (n > 0) {
        CU_TRY(c, cudaMemcpyAsync(c->d_pts1_raw, pts1, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
        CU_TRY(c, cudaMemcpyAsync(c->d_pts2_raw, pts2, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
    }
    launch_clip_points(c->stream, c->d_pts1_raw, c->d_pts1, n, c->w, c->h);
    launch_clip_points(c->stream, c->d_pts2_raw, c->d_pts2, n, c->w, c->h);
    c->launches += 2; c->class_launches[KC_MISC] += 2;
    CU_TRY(c, cudaGetLastError());
    CU_TRY(c, cudaStreamSynchronize(c->stream));   // the host arrays may be pageable and reused by the caller
    c->n_points = n;
    c->have_points = true;
    return 0;
}

int poppy_cuda_render(poppy_cuda_ctx* c, int n_frames, const float* shape, const double* mask, const int32_t* tri_idx,
                      const int32_t* tri_off, int chain) {
    return poppy_cuda_render_range(c, 0, n_frames, shape, mask, tri_idx, tri_off, chain);
}

namespace {
int validate_plan(poppy_cuda_ctx* c, const int32_t* tri_idx, const int32_t* tri_off, int n_frames) {
    for (int f = 0; f < n_frames; ++f) {
        const int nt = tri_off[f + 1] - tri_off[f];
        if (nt < 0 || nt > c->max_tri) return fail(c, POPPY_CUDA_ERR_CAPACITY, "frame %d has %d triangles (max %d)", f, nt, c->max_tri);
        const int32_t* src = tri_idx + (size_t)tri_off[f] * 3;
        for (int j = 0; j < nt * 3; ++j)
            if ((unsigned)src[j] >= (unsigned)c->n_points)
                return fail(c, POPPY_CUDA_ERR_INVALID, "frame %d: vertex index %d out of range [0,%d)", f, src[j], c->n_points);
    }
    return 0;
}
int render_impl(poppy_cuda_ctx* c, int first_slot, int n_frames, const float* shape, const double* mask, const int32_t* tri_idx,
                const int32_t* tri_off, int chain);
}  // namespace

int poppy_cuda_set_plan(poppy_cuda_ctx* c, const int32_t* tri_idx, const int32_t* tri_off, int n_frames) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (!c->have_points) return fail(c, POPPY_CUDA_ERR_STATE, "set_points must precede set_plan (vertex indices are checked against it)");
    if (!tri_off || n_frames < 1) return fail(c, POPPY_CUDA_ERR_INVALID, "bad plan");
    const size_t total = (size_t)(tri_off[n_frames] - tri_off[0]);
    if (!tri_idx && total) return fail(c, POPPY_CUDA_ERR_INVALID, "null triangle list");
    CU_TRY(c, cudaSetDevice(c->device));
    if (int rc = validate_plan(c, tri_idx, tri_off, n_frames)) return rc;
    // nothing queued may still read the plan it replaces
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    for (auto& l : c->lane) if (l.stream) CU_TRY(c, cudaStreamSynchronize(l.stream));
    if (total > c->plan_cap) {
        cudaFree(c->d_plan_tri);
        c->d_plan_tri = nullptr;
        c->plan_cap = 0;
        CU_TRY(c, dmalloc(&c->d_plan_tri, total));
        c->plan_cap = total;
    }
    if (total)
        CU_TRY(c, cudaMemcpy(c->d_plan_tri, tri_idx + (size_t)tri_off[0] * 3, total * sizeof(int3), cudaMemcpyHostToDevice));
    c->plan_off.resize((size_t)n_frames + 1);
    for (int f = 0; f <= n_frames; ++f) c->plan_off[f] = tri_off[f] - tri_off[0];
    c->plan_points = c->n_points;
    return 0;
}

int poppy_cuda_render_planned(poppy_cuda_ctx* c, int first_slot, int plan_first, int n_frames, const float* shape, const double* mask,
                              int chain) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (c->plan_off.empty() || c->plan_points != c->n_points)
        return fail(c, POPPY_CUDA_ERR_STATE, "no resident plan for the current point set (poppy_cuda_set_plan after set_points)");
    if (plan_first < 0 || n_frames < 1 || (size_t)plan_first + (size_t)n_frames > c->plan_off.size() - 1)
        return fail(c, POPPY_CUDA_ERR_INVALID, "frames [%d, %d) are not in the resident plan (%d frames)", plan_first, plan_first + n_frames,
                    (int)c->plan_off.size() - 1);
    return render_impl(c, first_slot, n_frames, shape, mask, nullptr, c->plan_off.data() + plan_first, chain);
}

int poppy_cuda_render_range(poppy_cuda_ctx* c, int first_slot, int n_frames, const float* shape, const double* mask,
                            const int32_t* tri_idx, const int32_t* tri_off, int chain) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (!tri_off) return fail(c, POPPY_CUDA_ERR_INVALID, "null argument");
    if (!tri_idx && n_frames >= 1 && tri_off[n_frames] != tri_off[0]) return fail(c, POPPY_CUDA_ERR_INVALID, "null triangle list");
    if (n_frames >= 1 && tri_idx) {
        // validate every frame before anything is enqueued: a failure must not leave earlier chunks running on the lanes
        if (!c->have_points) return fail(c, POPPY_CUDA_ERR_STATE, "set_pair and set_points must precede render");
        if (int rc = validate_plan(c, tri_idx, tri_off, n_frames)) return rc;
    }
    // an empty triangle list still needs a non-null base for the chunk staging
    static const int32_t none[3] = {0, 0, 0};
    return render_impl(c, first_slot, n_frames, shape, mask, tri_idx ? tri_idx : none, tri_off, chain);
}

namespace {
int render_impl(poppy_cuda_ctx* c, int first_slot, int n_frames, const float* shape, const double* mask, const int32_t* tri_idx,
                const int32_t* tri_off, int chain) {
    if (first_slot < 0) return fail(c, POPPY_CUDA_ERR_INVALID, "bad first_slot %d", first_slot);
    if (chain && first_slot > 0 && c->chain_next_slot != first_slot)
        return fail(c, POPPY_CUDA_ERR_STATE, "a chain continues at the slot after its last rendered frame (%d), not at %d", c->chain_next_slot, first_slot);
    if (!c->have_pair || !c->have_points) return fail(c, POPPY_CUDA_ERR_STATE, "set_pair and set_points must precede render");
    if (!shape || !mask || !tri_off) return fail(c, POPPY_CUDA_ERR_INVALID, "null argument");
    if (n_frames < 1 || first_slot + n_frames > c->max_frames)
        return fail(c, POPPY_CUDA_ERR_CAPACITY, "frames [%d, %d) exceed the ring (max %d)", first_slot, first_slot + n_frames, c->max_frames);
    CU_TRY(c, cudaSetDevice(c->device));
    if (int rc = ensure_chunk(c)) return rc;
    if (first_slot < c->copy_hi && first_slot + n_frames > c->copy_lo)      // slots with a download in flight
        CU_TRY(c, cudaStreamWaitEvent(c->stream, c->ev_copied, 0));
    collect_timing(c);
    std::fill(c->class_ms, c->class_ms + KC_COUNT, 0.f);
    std::fill(c->class_launches, c->class_launches + KC_COUNT, 0ull);
    // The context's stream brackets the render: the lanes start after everything queued on it so far (uploads, earlier
    // renders, downloads) and it continues after both lanes are done.
    CU_TRY(c, cudaEventRecord(c->ev_begin, c->stream));
    const int lanes = (chain || c->stage_timing) ? 1 : c->n_lanes;     // a chain is sequential; stage timing serialises
    for (int i = 0; i < lanes; ++i) CU_TRY(c, cudaStreamWaitEvent(c->lane[i].stream, c->ev_begin, 0));
    const int B = chain ? 1 : c->chunk;
    int k = 0;
    for (int first = 0; first < n_frames; first += B, ++k) {
        const int nb = std::min(B, n_frames - first);
        if (int rc = render_chunk(c, first_slot, first, nb, shape, mask, tri_idx, tri_off, chain != 0, c->lane[k % lanes])) {
            // a CUDA failure mid-render: still join the lanes so that later syncs / frees cover what was enqueued
            for (int i = 0; i < lanes; ++i) {
                cudaEventRecord(c->lane[i].ev_done, c->lane[i].stream);
                cudaStreamWaitEvent(c->stream, c->lane[i].ev_done, 0);
            }
            cudaEventRecord(c->ev_end, c->stream);
            return rc;
        }
    }
    for (int i = 0; i < lanes; ++i) {
        CU_TRY(c, cudaEventRecord(c->lane[i].ev_done, c->lane[i].stream));
        CU_TRY(c, cudaStreamWaitEvent(c->stream, c->lane[i].ev_done, 0));
    }
    CU_TRY(c, cudaEventRecord(c->ev_end, c->stream));
    c->last_frames = first_slot + n_frames;
    c->chain_next_slot = chain ? first_slot + n_frames : -1;
    c->seg_next_step = -1;          // the ring slots and points a segment render would continue from may be overwritten
    return 0;
}

}  // namespace

int poppy_cuda_set_segments(poppy_cuda_ctx* c, int n_segments, int window) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (n_segments < 1) return fail(c, POPPY_CUDA_ERR_INVALID, "n_segments must be >= 1");
    if (window < 2) return fail(c, POPPY_CUDA_ERR_INVALID, "window %d < 2: step j-1's points must survive step j", window);
    if ((long long)n_segments * window > c->max_frames)
        return fail(c, POPPY_CUDA_ERR_CAPACITY, "%d segments x %d slots exceed the ring (max %d)", n_segments, window, c->max_frames);
    CU_TRY(c, cudaSetDevice(c->device));
    // nothing queued may still read the segments being replaced
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    for (auto& l : c->lane) if (l.stream) CU_TRY(c, cudaStreamSynchronize(l.stream));
    free_segments(c);
    c->seg.resize(n_segments);
    for (auto& S : c->seg)
        for (int i = 0; i < 3; ++i)
            if (cudaError_t e = make_source_array(c->w, c->h, &S.a[i], &S.t[i])) {
                free_segments(c);
                return fail(c, POPPY_CUDA_ERR_CUDA, "segment source array: %s", cudaGetErrorString(e));
            }
    const size_t K = (size_t)n_segments, P = (size_t)c->max_points;
    if (dmalloc(&c->d_seg_basis, K * c->padded_pixels()) != cudaSuccess || dmalloc(&c->d_seg_raw, 2 * K * P) != cudaSuccess ||
        dmalloc(&c->d_seg_pts1, K * P) != cudaSuccess || dmalloc(&c->d_seg_pts2, K * P) != cudaSuccess) {
        free_segments(c);
        return fail(c, POPPY_CUDA_ERR_CUDA, "cannot allocate the resident data of %d segments", n_segments);
    }
    c->seg_window = window;
    return 0;
}

int poppy_cuda_set_segment(poppy_cuda_ctx* c, int s, const uint8_t* bgr1, size_t step1, const uint8_t* bgr2, size_t step2,
                           const float* gabor, size_t gstep, const float* pts1, const float* pts2, int n) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (s < 0 || s >= (int)c->seg.size()) return fail(c, POPPY_CUDA_ERR_INVALID, "segment %d not in [0,%d)", s, (int)c->seg.size());
    if (!bgr1 || !bgr2) return fail(c, POPPY_CUDA_ERR_INVALID, "null image pointer");
    const size_t row = (size_t)c->w * 3;
    if (step1 < row || step2 < row || (gabor && gstep < row * sizeof(float)))
        return fail(c, POPPY_CUDA_ERR_INVALID, "row stride smaller than a row");
    if ((n > 0 && (!pts1 || !pts2)) || n < 0) return fail(c, POPPY_CUDA_ERR_INVALID, "bad point sets");
    if (n > c->max_points) return fail(c, POPPY_CUDA_ERR_CAPACITY, "%d points (max %d)", n, c->max_points);
    CU_TRY(c, cudaSetDevice(c->device));
    if (int rc = ensure_pair_staging(c, 0)) return rc;
    if (gabor) if (int rc = ensure_pair_staging(c, 2)) return rc;
    poppy_cuda_ctx::Segment& S = c->seg[s];
    S.set = false;
    c->seg_next_step = -1;          // a chain cannot continue across a change of its inputs
    float* basis = c->d_seg_basis + (size_t)s * c->padded_pixels();
    if (int rc = upload_source(c, bgr1, step1, S.a[0])) return rc;
    if (int rc = upload_source(c, bgr2, step2, S.a[1])) return rc;
    if (!gabor) {
        // corrected2 is still in the 8-bit staging (same stream): the mask basis from it, as poppy_cuda_set_image(3)
        Scope sc(c, KC_MISC, c->stream);
        CU_TRY(c, launch_gabor_mask_basis(c->stream, c->d_stage_u8, basis, c->pitch0(), c->w, c->h));
    } else {
        CU_TRY(c, cudaMemcpy2DAsync(c->d_stage_f32, row * sizeof(float), gabor, gstep, row * sizeof(float), c->h,
                                    cudaMemcpyHostToDevice, c->stream));
        Scope sc(c, KC_MISC, c->stream);
        launch_mask_basis(c->stream, c->d_stage_f32, basis, c->pitch0(), c->w, c->h);
    }
    const size_t P = (size_t)c->max_points;
    float2* raw = c->d_seg_raw + 2 * (size_t)s * P;
    if (n > 0) {
        CU_TRY(c, cudaMemcpyAsync(raw, pts1, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
        CU_TRY(c, cudaMemcpyAsync(raw + P, pts2, (size_t)n * 8, cudaMemcpyHostToDevice, c->stream));
    }
    launch_clip_points(c->stream, raw, c->d_seg_pts1 + (size_t)s * P, n, c->w, c->h);
    launch_clip_points(c->stream, raw + P, c->d_seg_pts2 + (size_t)s * P, n, c->w, c->h);
    c->launches += 2; c->class_launches[KC_MISC] += 2;
    CU_TRY(c, cudaGetLastError());
    CU_TRY(c, cudaStreamSynchronize(c->stream));   // the host arrays may be pageable and reused by the caller
    S.n = n;
    S.set = true;
    return 0;
}

int poppy_cuda_render_segments(poppy_cuda_ctx* c, int first_step, int n_steps, const float* shape, const double* mask,
                               const int32_t* tri_idx, const int32_t* tri_off) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    const int K = (int)c->seg.size(), W = c->seg_window;
    if (K == 0) return fail(c, POPPY_CUDA_ERR_STATE, "poppy_cuda_set_segments must precede render_segments");
    for (int s = 0; s < K; ++s)
        if (!c->seg[s].set) return fail(c, POPPY_CUDA_ERR_STATE, "segment %d has not been set (poppy_cuda_set_segment)", s);
    if (c->keep_stages) return fail(c, POPPY_CUDA_ERR_STATE, "segment renders keep no stage buffers (set_keep_stages(0))");
    if (first_step < 0 || n_steps < 1) return fail(c, POPPY_CUDA_ERR_INVALID, "bad step range [%d, %d)", first_step, first_step + n_steps);
    if (first_step > 0 && first_step != c->seg_next_step)
        return fail(c, POPPY_CUDA_ERR_STATE, "a segment render continues at the step after its last rendered one (%d), not at %d",
                    c->seg_next_step, first_step);
    if (!shape || !mask || !tri_off) return fail(c, POPPY_CUDA_ERR_INVALID, "null argument");
    const int entries = n_steps * K;
    if (!tri_idx && tri_off[entries] != tri_off[0]) return fail(c, POPPY_CUDA_ERR_INVALID, "null triangle list");
    // validate every list against its own segment's points before anything is enqueued
    for (int e = 0; e < entries; ++e) {
        const int s = e % K, nt = tri_off[e + 1] - tri_off[e];
        if (nt < 0 || nt > c->max_tri)
            return fail(c, POPPY_CUDA_ERR_CAPACITY, "step %d of segment %d has %d triangles (max %d)", first_step + e / K, s, nt, c->max_tri);
        const int32_t* src = tri_idx ? tri_idx + (size_t)tri_off[e] * 3 : nullptr;
        for (int j = 0; j < nt * 3; ++j)
            if ((unsigned)src[j] >= (unsigned)c->seg[s].n)
                return fail(c, POPPY_CUDA_ERR_INVALID, "step %d of segment %d: vertex index %d out of range [0,%d)", first_step + e / K, s,
                            src[j], c->seg[s].n);
    }
    static const int32_t none[3] = {0, 0, 0};
    if (!tri_idx) tri_idx = none;
    CU_TRY(c, cudaSetDevice(c->device));
    if (int rc = ensure_chunk(c)) return rc;
    const int G = std::min(c->chunk, K);            // segments per group
    if (int rc = ensure_seg_lanes(c, G)) return rc;
    if (c->copy_hi > c->copy_lo && c->copy_lo < K * W)       // slots with a download in flight
        CU_TRY(c, cudaStreamWaitEvent(c->stream, c->ev_copied, 0));
    collect_timing(c);
    std::fill(c->class_ms, c->class_ms + KC_COUNT, 0.f);
    std::fill(c->class_launches, c->class_launches + KC_COUNT, 0ull);
    CU_TRY(c, cudaEventRecord(c->ev_begin, c->stream));
    // every step of a group runs on one lane (its chain is a recurrence); the groups go round-robin over the lanes
    const int lanes = c->stage_timing ? 1 : c->n_lanes;
    for (int i = 0; i < lanes; ++i) CU_TRY(c, cudaStreamWaitEvent(c->lane[i].stream, c->ev_begin, 0));
    int rc = 0;
    c->seg_next_step = -1;
    for (int r = 0; r < n_steps && !rc; ++r)
        for (int g = 0; g * G < K && !rc; ++g) {
            const SegChunk sg{g * G, first_step + r, r};
            rc = render_chunk(c, 0, 0, std::min(G, K - g * G), shape, mask, tri_idx, tri_off, true, c->lane[g % lanes], &sg);
        }
    for (int i = 0; i < lanes; ++i) {
        cudaEventRecord(c->lane[i].ev_done, c->lane[i].stream);
        cudaStreamWaitEvent(c->stream, c->lane[i].ev_done, 0);
    }
    cudaEventRecord(c->ev_end, c->stream);
    if (rc) return rc;
    CU_TRY(c, cudaGetLastError());
    c->chain_next_slot = -1;        // the pair's chain slots are overwritten
    c->last_frames = 0;
    c->seg_next_step = first_step + n_steps;
    return 0;
}

int poppy_cuda_get_segment_points(poppy_cuda_ctx* c, int s, int step, float* xy) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (!xy || s < 0 || s >= (int)c->seg.size()) return fail(c, POPPY_CUDA_ERR_INVALID, "bad segment %d or null pointer", s);
    const int W = c->seg_window;
    if (c->seg_next_step < 0 || step >= c->seg_next_step || step < std::max(0, c->seg_next_step - W))
        return fail(c, POPPY_CUDA_ERR_INVALID, "step %d of segment %d is not in the ring", step, s);
    CU_TRY(c, cudaSetDevice(c->device));
    if (c->seg[s].n > 0)
        CU_TRY(c, cudaMemcpyAsync(xy, c->d_morphed + ((size_t)s * W + step % W) * c->max_points, (size_t)c->seg[s].n * 8,
                                  cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return 0;
}

namespace {

// Downloads run after everything queued on the context's stream so far (the renders that produce their slots), but on the
// copy stream: later renders of other slots are not held up by the transfer.
int copy_after_renders(poppy_cuda_ctx* c) {
    CU_TRY(c, cudaEventRecord(c->ev_rendered, c->stream));
    CU_TRY(c, cudaStreamWaitEvent(c->copy_stream, c->ev_rendered, 0));
    return 0;
}

// After the copy-stream work of a download of slots [first, first + count): a later render of those slots waits for it.
int copies_enqueued(poppy_cuda_ctx* c, int first, int count) {
    CU_TRY(c, cudaEventRecord(c->ev_copied, c->copy_stream));
    if (c->copy_hi <= c->copy_lo) { c->copy_lo = first; c->copy_hi = first + count; }
    else { c->copy_lo = std::min(c->copy_lo, first); c->copy_hi = std::max(c->copy_hi, first + count); }
    return 0;
}

int issue_ticket(poppy_cuda_ctx* c, uint64_t* ticket) {
    if (c->tickets.empty()) {
        c->tickets.resize(64, nullptr);
        for (auto& e : c->tickets) CU_TRY(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    const uint64_t t = c->next_ticket++;
    CU_TRY(c, cudaEventRecord(c->tickets[t % c->tickets.size()], c->copy_stream));
    *ticket = t;
    return 0;
}

}  // namespace

int poppy_cuda_download(poppy_cuda_ctx* c, int first, int count, uint8_t* dst, size_t step, size_t frame_stride) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    const size_t row = (size_t)c->w * 3;
    if (!dst || first < 0 || count < 1 || first + count > c->max_frames || step < row || frame_stride < step * c->h)
        return fail(c, POPPY_CUDA_ERR_INVALID, "bad download range or strides");
    CU_TRY(c, cudaSetDevice(c->device));
    if (int rc = copy_after_renders(c)) return rc;
    if (step == row && frame_stride == c->frame_bytes()) {
        CU_TRY(c, cudaMemcpyAsync(dst, c->d_frames + (size_t)first * c->frame_bytes(), (size_t)count * c->frame_bytes(),
                                  cudaMemcpyDeviceToHost, c->copy_stream));
    } else {
        for (int i = 0; i < count; ++i)
            CU_TRY(c, cudaMemcpy2DAsync(dst + (size_t)i * frame_stride, step, c->d_frames + (size_t)(first + i) * c->frame_bytes(),
                                        row, row, c->h, cudaMemcpyDeviceToHost, c->copy_stream));
    }
    return copies_enqueued(c, first, count);
}

int poppy_cuda_download_i420(poppy_cuda_ctx* c, int first, int count, uint8_t* dst, size_t frame_stride) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if ((c->w | c->h) & 1)
        return fail(c, POPPY_CUDA_ERR_INVALID, "I420 needs an even frame size, the context's is %dx%d (cv::cvtColor throws too)",
                    c->w, c->h);
    const size_t fb = (size_t)c->w * c->h * 3 / 2;
    if (!dst) return fail(c, POPPY_CUDA_ERR_INVALID, "dst is null");
    if (first < 0 || count < 1 || first + count > c->max_frames)
        return fail(c, POPPY_CUDA_ERR_INVALID, "bad download range [%d, %d) of a %d-slot ring", first, first + count, c->max_frames);
    if (frame_stride < fb) return fail(c, POPPY_CUDA_ERR_INVALID, "frame_stride %zu is below the I420 frame size %zu", frame_stride, fb);
    CU_TRY(c, cudaSetDevice(c->device));
    if (!c->d_i420) {
        const int n = std::min(kI420StageFrames, c->max_frames);
        CU_TRY(c, cudaMalloc((void**)&c->d_i420, fb * n));
        c->i420_frames = n;
    }
    if (int rc = copy_after_renders(c)) return rc;
    // conversion and copy of each piece on the copy stream, in order: a piece's conversion overwrites the staging only after
    // the previous piece's copy has read it
    for (int done = 0; done < count; done += c->i420_frames) {
        const int n = std::min(c->i420_frames, count - done);
        launch_bgr_to_i420(c->copy_stream, c->d_frames, c->frame_bytes(), first + done, n, c->d_i420, c->w, c->h);
        c->launches++; c->class_launches[KC_MISC]++;
        CU_TRY(c, cudaGetLastError());
        if (frame_stride == fb) {
            CU_TRY(c, cudaMemcpyAsync(dst + (size_t)done * fb, c->d_i420, (size_t)n * fb, cudaMemcpyDeviceToHost, c->copy_stream));
        } else {
            for (int i = 0; i < n; ++i)
                CU_TRY(c, cudaMemcpyAsync(dst + (size_t)(done + i) * frame_stride, c->d_i420 + (size_t)i * fb, fb,
                                          cudaMemcpyDeviceToHost, c->copy_stream));
        }
    }
    return copies_enqueued(c, first, count);
}

int poppy_cuda_download_async(poppy_cuda_ctx* c, int first, int count, uint8_t* dst, size_t step, size_t frame_stride,
                              uint64_t* ticket) {
    if (!c || !ticket) return POPPY_CUDA_ERR_INVALID;
    if (int rc = poppy_cuda_download(c, first, count, dst, step, frame_stride)) return rc;
    return issue_ticket(c, ticket);
}

int poppy_cuda_download_i420_async(poppy_cuda_ctx* c, int first, int count, uint8_t* dst, size_t frame_stride, uint64_t* ticket) {
    if (!c || !ticket) return POPPY_CUDA_ERR_INVALID;
    if (int rc = poppy_cuda_download_i420(c, first, count, dst, frame_stride)) return rc;
    return issue_ticket(c, ticket);
}

namespace {

int ffv1_stage(poppy_cuda_ctx* c) {
    auto& f = c->ffv1;
    if (f.d_sym) return 0;
    poppy::ffv1::slice_grid(c->w, c->h, &f.nh, &f.nv);
    // at most 4096 frames a piece: the symbol kernel's grid z
    f.frames = (int)std::max<size_t>(1, std::min<size_t>({(size_t)c->max_frames, kFfv1StagePixels / c->pixels(), (size_t)4096}));
    const int slices = f.nh * f.nv * f.frames;
    // the largest slice: columns and rows are split as evenly as integer division allows
    const size_t slice_px = (size_t)((c->w + f.nh - 1) / f.nh) * ((c->h + f.nv - 1) / f.nv);
    f.cap = (slice_px * 3 + poppy::ffv1::kSliceAllowance + 15) / 16 * 16;                // raw sample bytes + allowance
    f.scratch_cap = (slice_px * poppy::ffv1::kWorstBytesPer3Samples + 2 * poppy::ffv1::kSliceAllowance + 15) / 16 * 16;
    uint8_t tables[512];
    poppy::ffv1::build_states(tables, tables + 256);
    CU_TRY(c, dmalloc(&f.d_sym, c->pixels() * 3 * f.frames));
    CU_TRY(c, dmalloc(&f.d_slots, f.cap * slices));
    f.packets_cap = f.cap * slices + (size_t)3 * slices;     // grows when slices are coded again into scratch
    CU_TRY(c, dmalloc(&f.d_packets, f.packets_cap));
    CU_TRY(c, dmalloc(&f.d_tables, 512));
    CU_TRY(c, dmalloc(&f.d_sizes, slices));
    CU_TRY(c, dmalloc(&f.d_frame_sizes, f.frames));
    CU_TRY(c, dmalloc(&f.d_offsets, slices + 1));
    CU_TRY(c, dmalloc(&f.d_slot_of, slices));
    CU_TRY(c, dmalloc(&f.d_overflow, slices + 1));
    CU_TRY(c, cudaMallocHost((void**)&f.h_overflow, sizeof(int)));
    CU_TRY(c, cudaMemcpy(f.d_tables, tables, 512, cudaMemcpyHostToDevice));
    return 0;
}

}  // namespace

int poppy_cuda_download_ffv1(poppy_cuda_ctx* c, int first, int count, uint8_t* dst, size_t cap, uint32_t* sizes) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (!dst || !sizes) return fail(c, POPPY_CUDA_ERR_INVALID, "dst or sizes is null");
    if (first < 0 || count < 1 || first + count > c->max_frames)
        return fail(c, POPPY_CUDA_ERR_INVALID, "bad download range [%d, %d) of a %d-slot ring", first, first + count, c->max_frames);
    CU_TRY(c, cudaSetDevice(c->device));
    if (int rc = ffv1_stage(c)) return rc;
    auto& f = c->ffv1;
    const int per_frame = f.nh * f.nv;
    if (int rc = copy_after_renders(c)) return rc;
    size_t total = 0;
    for (int done = 0; done < count; done += f.frames) {
        const int n = std::min(f.frames, count - done), slices = n * per_frame;
        launch_ffv1_symbols(c->copy_stream, c->d_frames, c->frame_bytes(), first + done, n, f.d_sym, c->w, c->h, f.nh, f.nv);
        CU_TRY(c, cudaMemsetAsync(f.d_overflow, 0, sizeof(int), c->copy_stream));
        CU_TRY(c, launch_ffv1_code(c->copy_stream, f.d_sym, f.d_tables, c->w, c->h, f.nh, f.nv, slices, nullptr, f.d_slots, f.cap,
                                   f.d_sizes, f.d_slot_of, f.d_overflow, f.d_overflow + 1));
        CU_TRY(c, cudaMemcpyAsync(f.h_overflow, f.d_overflow, sizeof(int), cudaMemcpyDeviceToHost, c->copy_stream));
        CU_TRY(c, cudaStreamSynchronize(c->copy_stream));
        const int over = *f.h_overflow;
        c->launches += 2; c->class_launches[KC_MISC] += 2;
        if (over > 0) {
            // slices whose samples did not fit their raw size are coded again, into worst-case scratch
            if ((size_t)over > f.scratch_slices) {
                CU_TRY(c, cudaFree(f.d_scratch));
                f.d_scratch = nullptr; f.scratch_slices = 0;
                CU_TRY(c, dmalloc(&f.d_scratch, f.scratch_cap * over));
                f.scratch_slices = over;
            }
            // the packets then hold up to `over` slices of scratch size
            const size_t need = (size_t)(slices - over) * f.cap + (size_t)over * f.scratch_cap + (size_t)3 * slices;
            if (need > f.packets_cap) {
                CU_TRY(c, cudaFree(f.d_packets));
                f.d_packets = nullptr; f.packets_cap = 0;
                CU_TRY(c, dmalloc(&f.d_packets, need));
                f.packets_cap = need;
            }
            CU_TRY(c, launch_ffv1_code(c->copy_stream, f.d_sym, f.d_tables, c->w, c->h, f.nh, f.nv, over, f.d_overflow + 1,
                                       f.d_scratch, f.scratch_cap, f.d_sizes, f.d_slot_of, f.d_overflow, f.d_overflow + 1));
            c->launches++; c->class_launches[KC_MISC]++;
        }
        launch_ffv1_pack(c->copy_stream, f.d_sizes, per_frame, n, f.d_offsets, f.d_frame_sizes, f.d_slots, f.cap, f.d_scratch,
                         f.scratch_cap, f.d_slot_of, f.d_packets);
        c->launches += 2; c->class_launches[KC_MISC] += 2;
        CU_TRY(c, cudaGetLastError());
        // only the packets cross PCIe: their sizes first, then exactly their bytes
        CU_TRY(c, cudaMemcpyAsync(sizes + done, f.d_frame_sizes, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, c->copy_stream));
        CU_TRY(c, cudaStreamSynchronize(c->copy_stream));
        size_t bytes = 0;
        for (int i = 0; i < n; ++i) bytes += sizes[done + i];
        if (total + bytes <= cap)
            CU_TRY(c, cudaMemcpyAsync(dst + total, f.d_packets, bytes, cudaMemcpyDeviceToHost, c->copy_stream));
        total += bytes;
    }
    if (int rc = copies_enqueued(c, first, count)) return rc;
    CU_TRY(c, cudaStreamSynchronize(c->copy_stream));
    if (total > cap)
        return fail(c, POPPY_CUDA_ERR_INVALID, "the %d packets take %zu bytes, dst holds %zu (sizes[] has each packet's size)", count,
                    total, cap);
    return 0;
}

int poppy_cuda_download_wait(poppy_cuda_ctx* c, uint64_t ticket) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (ticket >= c->next_ticket) return POPPY_CUDA_ERR_INVALID;
    // a ticket older than the pool is long complete: the copy stream is in order and its event slot has been re-recorded
    // by a later download, which can only finish after this one
    if (cudaSetDevice(c->device) != cudaSuccess || cudaEventSynchronize(c->tickets[ticket % c->tickets.size()]) != cudaSuccess)
        return POPPY_CUDA_ERR_CUDA;
    return 0;
}

int poppy_cuda_alloc_pinned(size_t bytes, void** out) {
    if (!out) return POPPY_CUDA_ERR_INVALID;
    *out = nullptr;
    return cudaMallocHost(out, bytes ? bytes : 1) == cudaSuccess ? 0 : POPPY_CUDA_ERR_CUDA;
}

void poppy_cuda_free_pinned(void* p) { if (p) cudaFreeHost(p); }

int poppy_cuda_get_morphed_points(poppy_cuda_ctx* c, int frame, float* xy) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (!xy || frame < 0 || frame >= c->last_frames) return fail(c, POPPY_CUDA_ERR_INVALID, "frame %d not rendered", frame);
    CU_TRY(c, cudaSetDevice(c->device));
    CU_TRY(c, cudaMemcpyAsync(xy, c->d_morphed + (size_t)frame * c->max_points, (size_t)c->n_points * 8,
                              cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int poppy_cuda_frame_device_ptr(poppy_cuda_ctx* c, int frame, void** dptr, size_t* bytes) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (!dptr || frame < 0 || frame >= c->max_frames) return fail(c, POPPY_CUDA_ERR_INVALID, "bad frame slot");
    *dptr = c->d_frames + (size_t)frame * c->frame_bytes();
    if (bytes) *bytes = c->frame_bytes();
    return 0;
}

int poppy_cuda_checksum(poppy_cuda_ctx* c, int first, int count, uint64_t* out) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (!out || first < 0 || count < 1 || first + count > c->max_frames) return fail(c, POPPY_CUDA_ERR_INVALID, "bad range");
    CU_TRY(c, cudaSetDevice(c->device));
    CU_TRY(c, cudaMemsetAsync(c->d_sum, 0, 8, c->stream));
    launch_checksum(c->stream, c->d_frames + (size_t)first * c->frame_bytes(), (size_t)count * c->frame_bytes(), c->d_sum);
    c->launches++; c->class_launches[KC_MISC]++;
    unsigned long long v = 0;
    CU_TRY(c, cudaMemcpyAsync(&v, c->d_sum, 8, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    *out = v;
    return 0;
}

int poppy_cuda_sync(poppy_cuda_ctx* c) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    CU_TRY(c, cudaSetDevice(c->device));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->copy_stream));
    c->copy_lo = c->copy_hi = 0;
    return 0;
}

int poppy_cuda_get_stream(poppy_cuda_ctx* c, void** stream) {
    if (!c || !stream) return POPPY_CUDA_ERR_INVALID;
    *stream = (void*)c->stream;
    return 0;
}

int poppy_cuda_last_render_ms(poppy_cuda_ctx* c, float* ms) {
    if (!c || !ms) return POPPY_CUDA_ERR_INVALID;
    CU_TRY(c, cudaSetDevice(c->device));
    CU_TRY(c, cudaEventSynchronize(c->ev_end));
    CU_TRY(c, cudaEventElapsedTime(ms, c->ev_begin, c->ev_end));
    return 0;
}

int poppy_cuda_launch_count(poppy_cuda_ctx* c, uint64_t* launches) {
    if (!c || !launches) return POPPY_CUDA_ERR_INVALID;
    *launches = c->launches;
    return 0;
}

int poppy_cuda_stage_times(poppy_cuda_ctx* c, const char** names, float* ms, uint64_t* launches, int cap) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    CU_TRY(c, cudaSetDevice(c->device));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    collect_timing(c);
    for (int i = 0; i < KC_COUNT && i < cap; ++i) {
        if (names) names[i] = kClassNames[i];
        if (ms) ms[i] = c->class_ms[i];
        if (launches) launches[i] = c->class_launches[i];
    }
    return KC_COUNT;
}

int poppy_cuda_debug_read(poppy_cuda_ctx* c, int stage, int frame, void* dst, size_t bytes) {
    if (!c) return POPPY_CUDA_ERR_INVALID;
    if (!dst) return fail(c, POPPY_CUDA_ERR_INVALID, "dst is null");
    if (stage == POPPY_STAGE_MASK_BASIS) {     // a property of the pair, not of a frame
        if (!c->keep_stages) return fail(c, POPPY_CUDA_ERR_STATE, "stage buffers need set_keep_stages(1)");
        if (!c->have_image[2]) return fail(c, POPPY_CUDA_ERR_STATE, "no mask basis: set_pair or set_image(2 or 3) first");
        if (bytes != c->pixels() * 4)
            return fail(c, POPPY_CUDA_ERR_INVALID, "stage %d holds %zu bytes, caller gave %zu", stage, c->pixels() * 4, bytes);
        CU_TRY(c, cudaSetDevice(c->device));
        CU_TRY(c, cudaStreamSynchronize(c->stream));
        CU_TRY(c, cudaMemcpy2D(dst, (size_t)c->w * 4, c->d_mbasis, (size_t)c->pitch0() * 4, (size_t)c->w * 4, c->h, cudaMemcpyDeviceToHost));
        return 0;
    }
    if (!c->keep_stages || c->chunk != 1) return fail(c, POPPY_CUDA_ERR_STATE, "stage buffers need set_keep_stages(1) before render");
    if (frame != c->last_frames - 1 && stage != POPPY_STAGE_MORPHED_POINTS)
        return fail(c, POPPY_CUDA_ERR_STATE, "only the last rendered frame's stage buffers are resident");
    CU_TRY(c, cudaSetDevice(c->device));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    const size_t px = c->pixels();
    const int w = c->w, h = c->h;
    FrameParams P;
    CU_TRY(c, cudaMemcpy(&P, c->lane[0].d_fp, sizeof P, cudaMemcpyDeviceToHost));
    auto need = [&](size_t want) -> int {
        return bytes == want ? 0 : fail(c, POPPY_CUDA_ERR_INVALID, "stage %d holds %zu bytes, caller gave %zu", stage, want, bytes);
    };
    switch (stage) {
    case POPPY_STAGE_MORPHED_POINTS:
        if (frame < 0 || frame >= c->last_frames) return fail(c, POPPY_CUDA_ERR_INVALID, "frame not rendered");
        if (int rc = need((size_t)c->n_points * 8)) return rc;
        CU_TRY(c, cudaMemcpy(dst, c->d_morphed + (size_t)frame * c->max_points, bytes, cudaMemcpyDeviceToHost));
        return 0;
    case POPPY_STAGE_TRI_MAP:
        if (int rc = need(px * 4)) return rc;
        CU_TRY(c, cudaMemcpy(dst, c->lane[0].d_trimap, bytes, cudaMemcpyDeviceToHost));
        return 0;
    case POPPY_STAGE_INV_M1:
    case POPPY_STAGE_INV_M2: {
        if (int rc = need((size_t)P.n_tri * 36)) return rc;
        std::vector<TriInverse> tmp(std::max(P.n_tri, 1));
        CU_TRY(c, cudaMemcpy(tmp.data(), c->lane[0].d_inv, (size_t)P.n_tri * sizeof(TriInverse), cudaMemcpyDeviceToHost));
        float* o = (float*)dst;
        for (int i = 0; i < P.n_tri; ++i) std::memcpy(o + 9 * i, stage == POPPY_STAGE_INV_M1 ? tmp[i].a : tmp[i].b, 36);
        return 0;
    }
    case POPPY_STAGE_WARPED1:
    case POPPY_STAGE_WARPED2: {
        if (int rc = need(px * 3)) return rc;
        std::vector<uint32_t> tmp(px);
        const uint32_t* plane = c->lane[0].d_warped + (stage == POPPY_STAGE_WARPED1 ? 0 : c->padded_pixels());
        CU_TRY(c, cudaMemcpy2D(tmp.data(), (size_t)w * 4, plane, (size_t)c->pitch0() * 4, (size_t)w * 4, h, cudaMemcpyDeviceToHost));
        uint8_t* o = (uint8_t*)dst;
        for (size_t i = 0; i < px; ++i) {
            uint32_t v = tmp[i];
            o[3 * i] = v & 255; o[3 * i + 1] = (v >> 8) & 255; o[3 * i + 2] = (v >> 16) & 255;
        }
        return 0;
    }
    case POPPY_STAGE_MASK:
        if (int rc = need(px * 4)) return rc;
        CU_TRY(c, cudaMemcpy2D(dst, (size_t)w * 4, c->lane[0].d_mask0, (size_t)c->pitch0() * 4, (size_t)w * 4, h, cudaMemcpyDeviceToHost));
        return 0;
    case POPPY_STAGE_LAP_BLEND: {
        if (int rc = need(px * 12)) return rc;
        const LevelDesc& d = c->lv[0];
        std::vector<float> tmp(3 * d.plane_stride);
        CU_TRY(c, cudaMemcpy(tmp.data(), o_level(c, c->lane[0], 0), tmp.size() * 4, cudaMemcpyDeviceToHost));
        float* o = (float*)dst;
        for (int y = 0; y < h; ++y)
            for (int x = 0; x < w; ++x)
                for (int ch = 0; ch < 3; ++ch) o[((size_t)y * w + x) * 3 + ch] = tmp[ch * d.plane_stride + (size_t)y * d.pitch + x];
        return 0;
    }
    default:
        return fail(c, POPPY_CUDA_ERR_INVALID, "unknown stage %d", stage);
    }
}

}  // extern "C"
