#include "morph_images.hpp"

#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstring>
#include <exception>
#include <map>
#include <memory>
#include <mutex>
#include <thread>
#include <utility>

#include "../../../include/poppy_host.h"

namespace poppy {

Settings* Settings::instance_ = nullptr;

namespace {

struct CachedContext {
    poppy_cuda_ctx* ctx = nullptr;
    int w = 0, h = 0, levels = 0, max_points = 0, max_tri = 0, max_frames = 0, device = 0;
    ~CachedContext() { if (ctx) poppy_cuda_destroy(ctx); }
};

std::mutex g_mu;
std::map<int, std::unique_ptr<CachedContext>> g_cached;   // by device

void cu(poppy_cuda_ctx* c, int rc) {
    if (rc != 0) throw MorphError(std::string("poppy_cuda: ") + poppy_cuda_last_error(c));
}

// the context cached in `slot` for `device`, recreated when the call needs another size or more capacity
poppy_cuda_ctx* context_in(std::unique_ptr<CachedContext>& slot, int device, int w, int h, int levels, int n_points, int n_tri,
                           int n_frames) {
    CachedContext* k = slot.get();
    if (k && k->w == w && k->h == h && k->levels == levels && k->device == device && k->max_points >= n_points &&
        k->max_tri >= n_tri && k->max_frames >= n_frames)
        return k->ctx;
    slot.reset(new CachedContext());
    k = slot.get();
    k->w = w; k->h = h; k->levels = levels; k->device = device;
    k->max_points = std::max(n_points, 64);
    k->max_tri = std::max(2 * n_points + 16, n_tri);
    k->max_frames = n_frames;
    int rc = poppy_cuda_create(&k->ctx, device, w, h, levels, k->max_points, k->max_tri, k->max_frames);
    if (rc != 0) {
        std::string msg = std::string("poppy_cuda_create: ") + poppy_cuda_last_error(nullptr);
        slot.reset();
        throw MorphError(msg);
    }
    // both entry points render one frame per kernel batch (a single frame, or a chain = a recurrence): size the scratch for
    // that instead of the 32-frame batches of direct-mode sequences
    poppy_cuda_set_chunk_frames(k->ctx, 1);
    return k->ctx;
}

poppy_cuda_ctx* context_for(int w, int h, int levels, int n_points, int n_tri, int n_frames) {
    const int device = Settings::instance().cuda_device;
    return context_in(g_cached[device], device, w, h, levels, n_points, n_tri, n_frames);
}

}  // namespace

void release_cached_contexts() {
    std::lock_guard<std::mutex> lock(g_mu);
    g_cached.clear();
}

double morph_images(const Image8& img1, const Image8& /*img2*/, const Image8& corrected1, const Image8& corrected2,
                    const Image32F& gabor2, Image8& /*goodFeatures1*/, Image8& /*goodFeatures2*/, Image8& dst,
                    const Image8& /*last*/, std::vector<Point2f>& morphedPoints, std::vector<Point2f> srcPoints1,
                    std::vector<Point2f> srcPoints2, double shapeRatio, double maskRatio, double /*linear*/) {
    const int w = img1.cols, h = img1.rows;
    if (corrected1.cols != w || corrected1.rows != h || corrected2.cols != w || corrected2.rows != h ||
        gabor2.cols != w || gabor2.rows != h)
        throw MorphError("morph_images: image sizes differ");
    // per frame, gabor2 is the caller's (the reference's signature); deriving it here would repeat the filter every frame
    if (!gabor2.data) throw MorphError("morph_images: gabor2 is empty");
    if (srcPoints1.size() != srcPoints2.size()) throw MorphError("morph_images: point sets differ in size");
    const int n = (int)srcPoints1.size();

    // host stages, reference src/algo.cpp:184-213 (subDiv1/subDiv2 feed only the GUI analysis and are skipped)
    clip_points(srcPoints1, w, h);
    clip_points(srcPoints2, w, h);
    morphedPoints.resize(n);
    static const float none[2] = {0.f, 0.f};
    const float* p1 = n ? &srcPoints1.data()->x : none;
    const float* p2 = n ? &srcPoints2.data()->x : none;
    float* mp = n ? &morphedPoints.data()->x : nullptr;
    if (n) poppy_host_morph_points(p1, p2, n, shapeRatio, w, h, mp);
    std::lock_guard<std::mutex> lock(g_mu);
    // sized for the most triangles n points can give, so that the pair can travel to the device while this thread triangulates
    poppy_cuda_ctx* c = context_for(w, h, (int)Settings::instance().pyramid_levels, n, 2 * n + 16, 1);
    int rc_up = 0;
    std::thread upload([&] {
        rc_up = poppy_cuda_set_pair(c, corrected1.data, corrected1.step, corrected2.data, corrected2.step, gabor2.data, gabor2.step);
        if (rc_up == 0) rc_up = poppy_cuda_set_points(c, p1, p2, n);
    });
    std::vector<int32_t> tri;
    std::string err;
    const bool tri_ok = triangulate_points_next(morphedPoints, w, h, tri, &err);
    upload.join();
    if (!tri_ok) throw MorphError("morph_images: " + err);
    cu(c, rc_up);
    const int n_tri = (int)tri.size() / 3;
    const float s = (float)shapeRatio;
    const int32_t offs[2] = {0, n_tri};
    cu(c, poppy_cuda_render(c, 1, &s, &maskRatio, tri.data(), offs, 0));
    if (dst.cols != w || dst.rows != h || dst.data == nullptr) dst.create(w, h);
    cu(c, poppy_cuda_download(c, 0, 1, dst.data, dst.step, dst.step * h));
    // the device recomputes morph_points(); hand back its copy (bit-identical to the host's, see tests)
    if (n) cu(c, poppy_cuda_get_morphed_points(c, 0, mp));
    cu(c, poppy_cuda_sync(c));
    return 0;
}

void morph_sequence(const Image8& corrected1, const Image8& corrected2, const Image32F& gabor2,
                    std::vector<Point2f> srcPoints1, std::vector<Point2f> srcPoints2, int number_of_frames,
                    const std::function<void(const Image8&)>& write) {
    const int w = corrected1.cols, h = corrected1.rows, n = (int)srcPoints1.size(), N = number_of_frames;
    if (N < 1) return;
    if (srcPoints1.size() != srcPoints2.size()) throw MorphError("morph_sequence: point sets differ in size");
    std::vector<float> ratio(N);
    std::vector<double> mask(N);
    for (int j = 0; j < N; ++j) { mask[j] = poppy_host_chain_ratio(j, N); ratio[j] = (float)mask[j]; }
    poppy_host_plan* plan = nullptr;
    static const float none[2] = {0.f, 0.f};
    const float* p1 = n ? &srcPoints1.data()->x : none;
    const float* p2 = n ? &srcPoints2.data()->x : none;
    if (poppy_host_plan_create(&plan, p1, p2, n, w, h, N, ratio.data(), 1, 0) != 0)
        throw MorphError(std::string("morph_sequence: ") + poppy_host_last_error());
    struct PlanGuard { poppy_host_plan* p; ~PlanGuard() { poppy_host_plan_destroy(p); } } guard{plan};
    const int32_t *tri = nullptr, *offs = nullptr;
    int max_tri = 0;
    poppy_host_plan_triangles(plan, &tri, &offs, &max_tri);

    std::lock_guard<std::mutex> lock(g_mu);
    poppy_cuda_ctx* c = context_for(w, h, (int)Settings::instance().pyramid_levels, n, max_tri, N);
    // gabor2.data == nullptr: set_pair derives the mask basis from corrected2
    cu(c, poppy_cuda_set_pair(c, corrected1.data, corrected1.step, corrected2.data, corrected2.step, gabor2.data, gabor2.step));
    cu(c, poppy_cuda_set_points(c, p1, p2, n));
    // The chain is rendered slice by slice (frame j-1 stays in HBM as frame j's source across the calls) and every finished
    // slice is handed to the writer ring: slice k+1 renders while slice k downloads and slice k-1 is being written.
    struct Sink { const std::function<void(const Image8&)>* write; } sink{&write};
    auto deliver = [](void* u, int, uint8_t* bgr, int fw, int fh, size_t step) {
        Image8 f;
        f.data = bgr; f.cols = fw; f.rows = fh; f.step = step;
        (*static_cast<Sink*>(u)->write)(f);
    };
    poppy_host_writer* wr = nullptr;
    if (poppy_host_writer_create(&wr, c, std::min(N, 8), deliver, nullptr, 0, &sink) != 0)
        throw MorphError("morph_sequence: cannot create the writer ring");
    struct WriterGuard { poppy_host_writer* w; ~WriterGuard() { poppy_host_writer_destroy_cuda(w); } } wguard{wr};
    const int S = 4;
    std::vector<int32_t> so;
    for (int a = 0; a < N; a += S) {
        const int cnt = std::min(S, N - a);
        so.assign(cnt + 1, 0);
        for (int i = 0; i <= cnt; ++i) so[i] = offs[a + i] - offs[a];
        cu(c, poppy_cuda_render_range(c, a, cnt, ratio.data() + a, mask.data() + a, tri + (size_t)offs[a] * 3, so.data(), 1));
        if (poppy_host_writer_submit(wr, a, cnt, a) != 0) throw MorphError(std::string("morph_sequence: ") + poppy_cuda_last_error(c));
    }
    if (poppy_host_writer_flush(wr) != 0) throw MorphError("morph_sequence: a frame download failed");
}

void morph_sequence(const Image8& corrected1, const Image8& corrected2, std::vector<Point2f> srcPoints1,
                    std::vector<Point2f> srcPoints2, int number_of_frames, const std::function<void(const Image8&)>& write) {
    morph_sequence(corrected1, corrected2, Image32F(), std::move(srcPoints1), std::move(srcPoints2), number_of_frames, write);
}

namespace {

// every segment's chain, planned as morph_sequence plans it
struct SegmentPlans {
    int N = 0, w = 0, h = 0, n_max = 0, tri_max = 0;
    std::vector<float> ratio;
    std::vector<double> mask;
    std::vector<poppy_host_plan*> p;
    std::vector<const int32_t*> tri, offs;
    ~SegmentPlans() { for (auto* q : p) poppy_host_plan_destroy(q); }
};

void plan_segments(const std::vector<Segment>& segments, int N, SegmentPlans& P) {
    const int K = (int)segments.size();
    const int w = segments[0].corrected1.cols, h = segments[0].corrected1.rows;
    for (const Segment& s : segments) {
        if (s.corrected1.cols != w || s.corrected1.rows != h || s.corrected2.cols != w || s.corrected2.rows != h)
            throw MorphError("morph_segments: all segments must have the same frame size");
        if (s.srcPoints1.size() != s.srcPoints2.size()) throw MorphError("morph_segments: point sets differ in size");
    }
    P.N = N; P.w = w; P.h = h;
    P.ratio.resize(N);
    P.mask.resize(N);
    for (int j = 0; j < N; ++j) { P.mask[j] = poppy_host_chain_ratio(j, N); P.ratio[j] = (float)P.mask[j]; }
    P.tri.resize(K);
    P.offs.resize(K);
    static const float none[2] = {0.f, 0.f};
    for (int s = 0; s < K; ++s) {
        const int n = (int)segments[s].srcPoints1.size();
        poppy_host_plan* plan = nullptr;
        if (poppy_host_plan_create(&plan, n ? &segments[s].srcPoints1.data()->x : none, n ? &segments[s].srcPoints2.data()->x : none,
                                   n, w, h, N, P.ratio.data(), 1, 0) != 0)
            throw MorphError("morph_segments: segment " + std::to_string(s) + ": " + poppy_host_last_error());
        P.p.push_back(plan);
        int mt = 0;
        poppy_host_plan_triangles(plan, &P.tri[s], &P.offs[s], &mt);
        P.n_max = std::max(P.n_max, n);
        P.tri_max = std::max(P.tri_max, mt);
    }
}

// Frames of several devices reach `write` in the output order: frame i is handed over once frames 0 .. i-1 have been.
// Each device delivers increasing indices of one contiguous range, so the device holding frame `next` always makes progress.
struct Turnstile {
    std::mutex mu;
    std::condition_variable cv;
    int next = 0;
    std::atomic<bool> failed{false};
};

struct Sink {
    const std::function<void(const Image8&)>* write;
    Turnstile* ts;
};

void deliver_in_turn(void* u, int index, uint8_t* bgr, int fw, int fh, size_t step) {
    Sink* k = static_cast<Sink*>(u);
    Turnstile& t = *k->ts;
    {
        std::unique_lock<std::mutex> lk(t.mu);
        t.cv.wait(lk, [&] { return t.failed || t.next == index; });
        if (t.failed) return;                  // another device failed: the call ends without writing more frames
    }
    Image8 f;
    f.data = bgr; f.cols = fw; f.rows = fh; f.step = step;
    (*k->write)(f);
    {
        std::lock_guard<std::mutex> lk(t.mu);
        ++t.next;
    }
    t.cv.notify_all();
}

// Segments [s0, s1) on one context, in batches of per_batch segments; segment s's step j is output frame s * N + j.
void render_share(poppy_cuda_ctx* c, poppy_host_writer* wr, const std::vector<Segment>& segments, const SegmentPlans& P, int s0,
                  int s1, int per_batch, Turnstile& ts) {
    static const float none[2] = {0.f, 0.f};
    const int N = P.N, S = 4;                          // steps per render call
    std::vector<int32_t> st, so;
    for (int b0 = s0; b0 < s1; b0 += per_batch) {
        const int kb = std::min(per_batch, s1 - b0);
        // The batch's first segment is written as it renders (its step j is ring slot j) when every earlier frame has been
        // written. Otherwise the writer ring would fill with frames waiting for their turn and hold this device's render
        // until the devices before it finish; the whole batch is then submitted after it has rendered.
        bool stream;
        {
            std::lock_guard<std::mutex> lk(ts.mu);
            stream = ts.next == b0 * N;
        }
        cu(c, poppy_cuda_set_segments(c, kb, N));
        for (int i = 0; i < kb; ++i) {
            const Segment& g = segments[b0 + i];
            const int n = (int)g.srcPoints1.size();
            cu(c, poppy_cuda_set_segment(c, i, g.corrected1.data, g.corrected1.step, g.corrected2.data, g.corrected2.step, g.gabor2.data,
                                         g.gabor2.step, n ? &g.srcPoints1.data()->x : none, n ? &g.srcPoints2.data()->x : none, n));
        }
        for (int a = 0; a < N; a += S) {
            if (ts.failed) return;
            const int cnt = std::min(S, N - a);
            // the slice's lists, step-major: entry r * kb + i is step a + r of segment b0 + i
            st.clear();
            so.assign(1, 0);
            for (int r = 0; r < cnt; ++r)
                for (int i = 0; i < kb; ++i) {
                    const int32_t* o = P.offs[b0 + i];
                    st.insert(st.end(), P.tri[b0 + i] + (size_t)o[a + r] * 3, P.tri[b0 + i] + (size_t)o[a + r + 1] * 3);
                    so.push_back((int32_t)(st.size() / 3));
                }
            cu(c, poppy_cuda_render_segments(c, a, cnt, P.ratio.data() + a, P.mask.data() + a, st.data(), so.data()));
            if (stream && poppy_host_writer_submit(wr, a, cnt, b0 * N + a) != 0)
                throw MorphError(std::string("morph_segments: ") + poppy_cuda_last_error(c));
        }
        for (int i = stream ? 1 : 0; i < kb; ++i)
            if (poppy_host_writer_submit(wr, i * N, N, (b0 + i) * N) != 0)
                throw MorphError(std::string("morph_segments: ") + poppy_cuda_last_error(c));
        // the next batch's segment data and frames replace this batch's: wait until every frame of it is written
        if (poppy_host_writer_flush(wr) != 0) throw MorphError("morph_segments: a frame download failed");
    }
}

// The segments over devices[0 .. G-1], G = min(devices.size(), K): device g renders the contiguous range
// [g * K / G, (g + 1) * K / G) (poppy_b200/shard.py phase_range) on its own cached context, driven by its own host thread
// (the calling thread drives devices[0]). Holds g_mu for the whole call.
void render_segments_on(const std::vector<Segment>& segments, int N, const std::function<void(const Image8&)>& write,
                        const std::vector<int>& devices) {
    const int K = (int)segments.size();
    if (K == 0 || N < 1) return;
    SegmentPlans P;
    plan_segments(segments, N, P);

    std::lock_guard<std::mutex> lock(g_mu);
    const int G = std::min((int)devices.size(), K);
    std::vector<std::unique_ptr<CachedContext>*> slots;          // resolved here: the threads must not insert into g_cached
    for (int g = 0; g < G; ++g) slots.push_back(&g_cached[devices[g]]);
    const int levels = (int)Settings::instance().pyramid_levels;
    Turnstile ts;
    Sink sink{&write, &ts};
    std::mutex err_mu;
    std::exception_ptr first_error;
    auto fail = [&](std::exception_ptr e) {
        {
            std::lock_guard<std::mutex> lk(err_mu);
            if (!first_error) first_error = e;
        }
        {
            std::lock_guard<std::mutex> lk(ts.mu);
            ts.failed = true;
        }
        ts.cv.notify_all();
    };
    auto run = [&](int g) {
        try {
            const int s0 = (int)((long long)g * K / G), s1 = (int)((long long)(g + 1) * K / G);
            // as many segments per batch as fit the device's ring at once (all N frames of each stay resident until written)
            const size_t frame_bytes = (size_t)P.w * P.h * 3, ring_bytes = 8ull << 30;
            const int per_batch = (int)std::max<size_t>(1, std::min<size_t>(s1 - s0, ring_bytes / (frame_bytes * N)));
            poppy_cuda_ctx* c = context_in(*slots[g], devices[g], P.w, P.h, levels, P.n_max, P.tri_max, per_batch * N);
            // a kernel batch holds one step of a group of segments; the cached context goes back to one frame per batch after
            cu(c, poppy_cuda_set_chunk_frames(c, std::min(per_batch, 32)));
            struct ChunkGuard { poppy_cuda_ctx* c; ~ChunkGuard() { poppy_cuda_set_chunk_frames(c, 1); } } cguard{c};
            poppy_host_writer* wr = nullptr;
            if (poppy_host_writer_create(&wr, c, std::min(N, 8), deliver_in_turn, nullptr, 0, &sink) != 0)
                throw MorphError("morph_segments: cannot create the writer ring");
            struct WriterGuard { poppy_host_writer* w; ~WriterGuard() { poppy_host_writer_destroy_cuda(w); } } wguard{wr};
            // caught here, before the writer's final flush: frames waiting for their turn are dropped instead of waited for
            try { render_share(c, wr, segments, P, s0, s1, per_batch, ts); }
            catch (...) { fail(std::current_exception()); }
        } catch (...) {
            fail(std::current_exception());
        }
    };
    std::vector<std::thread> threads;
    for (int g = 1; g < G; ++g) threads.emplace_back(run, g);
    run(0);
    for (auto& t : threads) t.join();
    if (first_error) std::rethrow_exception(first_error);
}

void check_devices(const std::vector<int>& devices) {
    if (devices.empty()) throw MorphError("morph_segments: the device list is empty");
    for (size_t i = 0; i < devices.size(); ++i) {
        if (devices[i] < 0) throw MorphError("morph_segments: device " + std::to_string(devices[i]) + " is negative");
        for (size_t j = 0; j < i; ++j)
            if (devices[j] == devices[i]) throw MorphError("morph_segments: device " + std::to_string(devices[i]) + " is listed twice");
    }
    const int n = poppy_cuda_device_count();
    if (n <= 0) throw NoDeviceError("morph_segments: no CUDA device: the morph renderer has no CPU fallback");
    for (int d : devices)
        if (d >= n) throw MorphError("morph_segments: device " + std::to_string(d) + " not in [0," + std::to_string(n) + ")");
}

}  // namespace

void morph_segments(const std::vector<Segment>& segments, int number_of_frames, const std::function<void(const Image8&)>& write) {
    render_segments_on(segments, number_of_frames, write, {Settings::instance().cuda_device});
}

void morph_segments(const std::vector<Segment>& segments, int number_of_frames, const std::function<void(const Image8&)>& write,
                    const std::vector<int>& devices) {
    check_devices(devices);
    render_segments_on(segments, number_of_frames, write, devices);
}

}  // namespace poppy
