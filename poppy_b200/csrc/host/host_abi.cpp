// extern "C" layer of the host stages (include/poppy_host.h).
#include <atomic>
#include <climits>
#include <cmath>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/poppy_host.h"
#include "delaunay.hpp"
#include "morph_images.hpp"

using poppy::Point2f;

namespace {
thread_local std::string g_host_error;

int host_fail(int code, const std::string& msg) {
    g_host_error = msg;
    return code;
}

// morph_points(), reference src/algo.cpp:50-58: the first product is double, the second float x float, the sum double
float lerp_coord(float a, float b, float s) {
    float sb = s * b;
    return (float)((1.0 - (double)s) * (double)a + (double)sb);
}

void lerp_points(const std::vector<Point2f>& a, const std::vector<Point2f>& b, float s, int w, int h,
                 std::vector<Point2f>& out) {
    out.resize(a.size());
    for (size_t i = 0; i < a.size(); ++i) out[i] = {lerp_coord(a[i].x, b[i].x, s), lerp_coord(a[i].y, b[i].y, s)};
    poppy::clip_points(out, w, h);
}

std::vector<Point2f> to_points(const float* xy, int n) {
    std::vector<Point2f> v(n);
    if (n) std::memcpy(v.data(), xy, (size_t)n * sizeof(Point2f));
    return v;
}
}  // namespace

struct poppy_host_plan {
    int n = 0, frames = 0, max_tri = 0;
    std::vector<std::vector<Point2f>> points;    // per frame
    std::vector<int32_t> tri;                    // concatenated
    std::vector<int32_t> offsets;                // frames + 1
};

// ---- the C++ shim (poppy::morph_images / poppy::morph_sequence, morph_images.hpp) behind C entry points ------------------
namespace {
template <class F> int shim_guard(F&& f) {
    try { f(); return 0; }
    catch (const poppy::NoDeviceError& e) { return host_fail(POPPY_CUDA_ERR_NO_DEVICE, e.what()); }
    catch (const poppy::MorphError& e) { return host_fail(POPPY_CUDA_ERR_INVALID, e.what()); }
    catch (const std::exception& e) { return host_fail(POPPY_CUDA_ERR_INVALID, e.what()); }
}
poppy::Image8 view8(const uint8_t* p, int w, int h, size_t step) {
    poppy::Image8 v;
    v.data = const_cast<uint8_t*>(p); v.cols = w; v.rows = h; v.step = step;
    return v;
}

int check_shim_segments(const poppy_shim_segment* segs, int n_segments, poppy_write_fn write) {
    if (!segs || !write || n_segments < 1) return host_fail(POPPY_CUDA_ERR_INVALID, "null argument");
    for (int s = 0; s < n_segments; ++s)
        if (!segs[s].corrected1 || !segs[s].corrected2 || segs[s].n < 0 || (segs[s].n > 0 && (!segs[s].pts1_xy || !segs[s].pts2_xy)))
            return host_fail(POPPY_CUDA_ERR_INVALID, "segment " + std::to_string(s) + ": null argument");
    return 0;
}

std::vector<poppy::Segment> shim_segments(int w, int h, const poppy_shim_segment* segs, int n_segments) {
    std::vector<poppy::Segment> v(n_segments);
    for (int s = 0; s < n_segments; ++s) {
        const poppy_shim_segment& g = segs[s];
        v[s].corrected1 = view8(g.corrected1, w, h, g.step1);
        v[s].corrected2 = view8(g.corrected2, w, h, g.step2);
        if (g.gabor2) { v[s].gabor2.data = g.gabor2; v[s].gabor2.cols = w; v[s].gabor2.rows = h; v[s].gabor2.step = g.gstep; }
        v[s].srcPoints1 = to_points(g.pts1_xy, g.n);
        v[s].srcPoints2 = to_points(g.pts2_xy, g.n);
    }
    return v;
}
}  // namespace

// The walk trace of the last frame a sequence planner call triangulated: it predicts the first frame of the next call.
namespace {
std::mutex g_trace_mutex;
poppy::WalkTrace g_carried_trace;
void take_carried_trace(poppy::WalkTrace& out) {
    std::lock_guard<std::mutex> lock(g_trace_mutex);
    std::swap(out, g_carried_trace);
    g_carried_trace.clear();
}
void put_carried_trace(poppy::WalkTrace& t) {
    std::lock_guard<std::mutex> lock(g_trace_mutex);
    std::swap(g_carried_trace, t);
}
}  // namespace

extern "C" {

const char* poppy_host_last_error(void) { return g_host_error.c_str(); }

int poppy_host_morph_points(const float* p1, const float* p2, int n, double shape_ratio, int w, int h, float* out) {
    if (!p1 || !p2 || !out || n < 0) return host_fail(POPPY_CUDA_ERR_INVALID, "null argument");
    std::vector<Point2f> a = to_points(p1, n), b = to_points(p2, n), m;
    poppy::clip_points(a, w, h);
    poppy::clip_points(b, w, h);
    lerp_points(a, b, (float)shape_ratio, w, h, m);
    if (n) std::memcpy(out, m.data(), (size_t)n * sizeof(Point2f));
    return 0;
}

int poppy_host_triangulate(const float* pts, int n, int w, int h, int32_t* tri_idx, int cap, int* n_tri) {
    if (!pts || !n_tri || n < 0) return host_fail(POPPY_CUDA_ERR_INVALID, "null argument");
    std::vector<int32_t> tri;
    std::string err;
    if (!poppy::triangulate_points(to_points(pts, n), w, h, tri, &err)) return host_fail(POPPY_CUDA_ERR_INVALID, err);
    *n_tri = (int)tri.size() / 3;
    if (*n_tri > cap) return host_fail(POPPY_CUDA_ERR_CAPACITY, "triangle buffer too small");
    if (tri_idx && !tri.empty()) std::memcpy(tri_idx, tri.data(), tri.size() * sizeof(int32_t));
    return 0;
}

int poppy_host_triangulate_next(const float* pts, int n, int w, int h, int32_t* tri_idx, int cap, int* n_tri) {
    if (!pts || !n_tri || n < 0) return host_fail(POPPY_CUDA_ERR_INVALID, "null argument");
    std::vector<int32_t> tri;
    std::string err;
    if (!poppy::triangulate_points_next(to_points(pts, n), w, h, tri, &err)) return host_fail(POPPY_CUDA_ERR_INVALID, err);
    *n_tri = (int)tri.size() / 3;
    if (*n_tri > cap) return host_fail(POPPY_CUDA_ERR_CAPACITY, "triangle buffer too small");
    if (tri_idx && !tri.empty()) std::memcpy(tri_idx, tri.data(), tri.size() * sizeof(int32_t));
    return 0;
}

double poppy_host_chain_ratio(int j, int n_frames) {
    // linear = j / N; progress = 0 for linear == 0, 1 for linear == 1, else (1 / (1 - linear)) / N; capped at 1
    const double N = (double)n_frames;
    const double linear = j / N;
    double progress;
    if (linear == 0) progress = 0;
    else if (linear == 1) progress = 1;
    else progress = (1.0 / (1.0 - linear)) / N;
    return progress > 1 ? 1 : progress;
}

int poppy_host_plan_create(poppy_host_plan** out, const float* p1, const float* p2, int n, int w, int h, int n_frames,
                           const float* shape_ratio, int chain, int threads) {
    if (!out) return host_fail(POPPY_CUDA_ERR_INVALID, "out is null");
    *out = nullptr;
    if (!p1 || !p2 || !shape_ratio || n < 0 || n_frames < 1) return host_fail(POPPY_CUDA_ERR_INVALID, "bad argument");
    poppy_host_plan* plan = new poppy_host_plan();
    plan->n = n;
    plan->frames = n_frames;
    plan->points.resize(n_frames);
    std::vector<Point2f> a = to_points(p1, n), b = to_points(p2, n);
    poppy::clip_points(a, w, h);
    poppy::clip_points(b, w, h);
    // points first: in chain mode frame f starts from frame f-1's morphed points (src/poppy.hpp:178-179); this
    // recurrence involves no pixels, so it is planned ahead of the render
    for (int f = 0; f < n_frames; ++f)
        lerp_points(chain && f > 0 ? plan->points[f - 1] : a, b, shape_ratio[f], w, h, plan->points[f]);
    // triangulations are independent: fan out over host threads
    std::vector<std::vector<int32_t>> tris(n_frames);
    std::vector<std::string> errs(n_frames);
    std::atomic<int> failed{-1};
    int nt = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    nt = std::max(1, std::min(nt, n_frames));
    // Worker t triangulates frames t, t + nt, t + 2 nt, ... Frame f is PREDICTED by frame f - 1 (poppy::WalkTrace), which
    // another worker is triangulating at the same time: frame f runs a few points behind it (poppy::WalkPace), so every
    // frame but the first is guided by its immediate neighbour - the distance at which the prediction is nearly perfect -
    // and all workers stay busy. Frame 0 is predicted by the last frame of the previous call (the previous slice of the
    // same sequence, typically); a stale guide costs its own mispredictions, never the result.
    const int ring = 2 * nt + 1;
    std::vector<poppy::WalkTrace> traces(ring);
    std::unique_ptr<std::atomic<int>[]> progress(new std::atomic<int>[n_frames + 1]);
    for (int f = 0; f <= n_frames; ++f) progress[f].store(0, std::memory_order_relaxed);
    poppy::WalkTrace carried;                                           // the previous call's last trace
    take_carried_trace(carried);
    std::atomic<int> worker_id{0};
    auto work = [&] {
        const int t = worker_id.fetch_add(1);
        for (int f = t; f < n_frames; f += nt) {
            // the ring slot of frame f was last used by frame f - ring, which frame f - ring + 1 was reading
            if (f - ring + 1 >= 0)
                while (progress[f - ring + 1].load(std::memory_order_acquire) != INT_MAX) std::this_thread::yield();
            poppy::WalkPace pace;
            pace.publish = &progress[f];
            pace.follow = f > 0 ? &progress[f - 1] : nullptr;
            const poppy::WalkTrace* guide = f > 0 ? &traces[(f - 1) % ring] : (carried.empty() ? nullptr : &carried);
            if (!poppy::triangulate_points(plan->points[f], w, h, tris[f], &errs[f], guide, &traces[f % ring], &pace)) {
                int expected = -1;
                failed.compare_exchange_strong(expected, f);
            }
        }
    };
    std::vector<std::thread> pool;
    for (int i = 1; i < nt; ++i) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
    put_carried_trace(traces[(n_frames - 1) % ring]);
    if (failed.load() >= 0) {
        std::string msg = "frame " + std::to_string(failed.load()) + ": " + errs[failed.load()];
        delete plan;
        return host_fail(POPPY_CUDA_ERR_INVALID, msg);
    }
    plan->offsets.assign(n_frames + 1, 0);
    for (int f = 0; f < n_frames; ++f) {
        const int t = (int)tris[f].size() / 3;
        plan->offsets[f + 1] = plan->offsets[f] + t;
        plan->max_tri = std::max(plan->max_tri, t);
    }
    // one contiguous list (the device ABI's layout); copied by the same number of threads - at 4K a 600-frame plan is 290 MB
    plan->tri.resize((size_t)plan->offsets[n_frames] * 3);
    {
        std::atomic<int> next_copy{0};
        auto copy = [&] {
            for (int f; (f = next_copy.fetch_add(1)) < n_frames;)
                if (!tris[f].empty())
                    std::memcpy(plan->tri.data() + (size_t)plan->offsets[f] * 3, tris[f].data(), tris[f].size() * sizeof(int32_t));
        };
        std::vector<std::thread> copiers;
        for (int i = 1; i < std::min(nt, 8); ++i) copiers.emplace_back(copy);
        copy();
        for (auto& t : copiers) t.join();
    }
    *out = plan;
    return 0;
}

int poppy_host_plan_triangles(const poppy_host_plan* plan, const int32_t** tri_idx, const int32_t** tri_offsets,
                              int* max_triangles) {
    if (!plan) return host_fail(POPPY_CUDA_ERR_INVALID, "plan is null");
    if (tri_idx) *tri_idx = plan->tri.data();
    if (tri_offsets) *tri_offsets = plan->offsets.data();
    if (max_triangles) *max_triangles = plan->max_tri;
    return 0;
}

int poppy_host_plan_points(const poppy_host_plan* plan, int frame, const float** xy) {
    if (!plan || !xy || frame < 0 || frame >= plan->frames) return host_fail(POPPY_CUDA_ERR_INVALID, "bad frame");
    *xy = &plan->points[frame][0].x;
    return 0;
}

void poppy_host_plan_destroy(poppy_host_plan* plan) { delete plan; }

int poppy_morph_images(poppy_cuda_ctx* ctx, const uint8_t* c1, size_t step1, const uint8_t* c2, size_t step2,
                       const float* gabor2, size_t gstep, const float* sp1, const float* sp2, int n,
                       double shape_ratio, double mask_ratio, uint8_t* dst, size_t dst_step, float* morphed_xy) {
    if (!ctx || !c1 || !c2 || !gabor2 || !dst || n < 0 || (n > 0 && (!sp1 || !sp2))) return host_fail(POPPY_CUDA_ERR_INVALID, "null argument");
    int w = 0, h = 0, max_tri = 0;
    if (int rc = poppy_cuda_get_info(ctx, &w, &h, nullptr, nullptr, &max_tri, nullptr)) return host_fail(rc, "bad context");
    // host stages, reference src/algo.cpp:184-213
    std::vector<Point2f> a = to_points(sp1, n), b = to_points(sp2, n), m;
    poppy::clip_points(a, w, h);
    poppy::clip_points(b, w, h);
    const float s = (float)shape_ratio;
    lerp_points(a, b, s, w, h, m);
    // the pair travels to the device (pageable host memory: ~150 MB at 4K) while this thread triangulates
    int rc_up = 0;
    std::thread upload([&] {
        rc_up = poppy_cuda_set_pair(ctx, c1, step1, c2, step2, gabor2, gstep);
        if (rc_up == 0) rc_up = poppy_cuda_set_points(ctx, sp1, sp2, n);
    });
    std::vector<int32_t> tri;
    std::string err;
    // the reference calls morph_images() once per frame of a sequence: the previous call's point-location walks predict this
    // call's (poppy::WalkTrace; any guide gives the same triangulation)
    const bool tri_ok = poppy::triangulate_points_next(m, w, h, tri, &err);
    upload.join();
    if (!tri_ok) return host_fail(POPPY_CUDA_ERR_INVALID, err);
    if (rc_up != 0) return host_fail(rc_up, poppy_cuda_last_error(ctx));
    const int32_t offs[2] = {0, (int32_t)(tri.size() / 3)};
    int rc;
    if ((rc = poppy_cuda_render(ctx, 1, &s, &mask_ratio, tri.data(), offs, 0)) != 0 ||
        (rc = poppy_cuda_download(ctx, 0, 1, dst, dst_step, dst_step * (size_t)h)) != 0 ||
        (morphed_xy && (rc = poppy_cuda_get_morphed_points(ctx, 0, morphed_xy)) != 0) ||
        (rc = poppy_cuda_sync(ctx)) != 0)
        return host_fail(rc, poppy_cuda_last_error(ctx));
    return 0;
}

int poppy_shim_morph_images(int w, int h, int pyramid_levels, const uint8_t* c1, size_t step1, const uint8_t* c2, size_t step2,
                            const float* gabor2, size_t gstep, const float* sp1, const float* sp2, int n, double shape_ratio,
                            double mask_ratio, uint8_t* dst, size_t dst_step, float* morphed_xy) {
    if (!c1 || !c2 || !gabor2 || !dst || n < 0 || (n > 0 && (!sp1 || !sp2))) return host_fail(POPPY_CUDA_ERR_INVALID, "null argument");
    return shim_guard([&] {
        poppy::Settings::instance().pyramid_levels = (size_t)pyramid_levels;
        poppy::Image8 img1 = view8(c1, w, h, step1), img2 = view8(c2, w, h, step2), none, out = view8(dst, w, h, dst_step);
        poppy::Image32F g;
        g.data = gabor2; g.cols = w; g.rows = h; g.step = gstep;
        std::vector<Point2f> a = to_points(sp1, n), b = to_points(sp2, n), m;
        poppy::morph_images(img1, img2, img1, img2, g, none, none, out, none, m, a, b, shape_ratio, mask_ratio, 0.0);
        if (morphed_xy && n) std::memcpy(morphed_xy, m.data(), (size_t)n * sizeof(Point2f));
    });
}

int poppy_shim_morph_sequence(int w, int h, int pyramid_levels, const uint8_t* c1, size_t step1, const uint8_t* c2, size_t step2,
                              const float* gabor2, size_t gstep, const float* sp1, const float* sp2, int n, int n_frames,
                              poppy_write_fn write, void* user) {
    if (!c1 || !c2 || !write || n < 0 || (n > 0 && (!sp1 || !sp2))) return host_fail(POPPY_CUDA_ERR_INVALID, "null argument");
    return shim_guard([&] {
        poppy::Settings::instance().pyramid_levels = (size_t)pyramid_levels;
        poppy::Image32F g;             // gabor2 == NULL: empty, derived on the device
        if (gabor2) { g.data = gabor2; g.cols = w; g.rows = h; g.step = gstep; }
        int index = 0;
        poppy::morph_sequence(view8(c1, w, h, step1), view8(c2, w, h, step2), g, to_points(sp1, n), to_points(sp2, n), n_frames,
                              [&](const poppy::Image8& f) { write(user, index++, f.data, f.cols, f.rows, f.step); });
    });
}

int poppy_shim_morph_segments(int w, int h, int pyramid_levels, const poppy_shim_segment* segs, int n_segments, int n_frames,
                              poppy_write_fn write, void* user) {
    if (int rc = check_shim_segments(segs, n_segments, write)) return rc;
    return shim_guard([&] {
        poppy::Settings::instance().pyramid_levels = (size_t)pyramid_levels;
        int index = 0;
        poppy::morph_segments(shim_segments(w, h, segs, n_segments), n_frames,
                              [&](const poppy::Image8& f) { write(user, index++, f.data, f.cols, f.rows, f.step); });
    });
}

int poppy_shim_morph_segments_devices(const int* devices, int n_devices, int w, int h, int pyramid_levels, const poppy_shim_segment* segs,
                                      int n_segments, int n_frames, poppy_write_fn write, void* user) {
    if (!devices || n_devices < 1) return host_fail(POPPY_CUDA_ERR_INVALID, "no devices");
    if (int rc = check_shim_segments(segs, n_segments, write)) return rc;
    return shim_guard([&] {
        poppy::Settings::instance().pyramid_levels = (size_t)pyramid_levels;
        int index = 0;
        poppy::morph_segments(shim_segments(w, h, segs, n_segments), n_frames,
                              [&](const poppy::Image8& f) { write(user, index++, f.data, f.cols, f.rows, f.step); },
                              std::vector<int>(devices, devices + n_devices));
    });
}

void poppy_shim_release(void) { poppy::release_cached_contexts(); }

}  // extern "C"
