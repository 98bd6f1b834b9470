// Writer hand-off (include/poppy_host.h, poppy_host_writer_*): the reference's frame loop passes every finished frame to
// Twriter::write(Mat&) (reference src/poppy.hpp:219: cv::VideoWriter on native builds, src/poppy.cpp:249; the GIF writer
// on WASM, src/poppy.cpp:57-84) and waits for it. Here the frames leave the GPU through a ring of page-locked buffers:
// the caller's thread enqueues the download of rendered ring slots and goes on planning / rendering, a delivery thread
// waits for each copy and calls `write` strictly in frame order (video encoders are order dependent), and an optional
// worker pool runs a per-frame `convert` step (pixel-format conversion, compression ...) ahead of delivery.
#include <atomic>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/poppy_host.h"

struct poppy_host_writer {
    poppy_host_writer_io io{};
    int width = 0, height = 0, ring = 0, workers = 0;
    size_t row_bytes = 0, frame_bytes = 0;      // of one ring buffer: BGR rows (width * 3), or the Y rows of an I420 frame
    std::vector<uint8_t*> buffers;              // page-locked frame buffers
    struct Item { int frame_index; int buffer; uint64_t ticket; bool converted; };
    std::mutex mu;
    std::condition_variable cv_free, cv_work, cv_done;
    std::deque<int> free_buffers;
    std::deque<Item> pending;                   // submitted, in frame order
    size_t next_convert = 0;                    // first entry of `pending` no worker has taken yet
    uint64_t submitted = 0, written = 0;
    bool stop = false, owned_ffv1 = false;     // owned_ffv1: io.owned_transport is an FFV1 transport
    int error = 0;
    std::thread deliverer;
    std::vector<std::thread> pool;

    void deliver_loop() {
        for (;;) {
            Item it;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_work.wait(lk, [&] { return stop || (!pending.empty() && (workers == 0 || pending.front().converted)); });
                if (pending.empty()) { if (stop) return; continue; }
                if (workers > 0 && !pending.front().converted) { if (stop) return; continue; }
                it = pending.front();
            }
            if (workers == 0) {
                if (io.wait && io.wait(io.user, it.ticket) != 0) { std::lock_guard<std::mutex> lk(mu); error = POPPY_CUDA_ERR_CUDA; }
            }
            if (io.write) io.write(io.user, it.frame_index, buffers[it.buffer], width, height, row_bytes);
            {
                std::lock_guard<std::mutex> lk(mu);
                pending.pop_front();
                if (next_convert > 0) --next_convert;
                free_buffers.push_back(it.buffer);
                ++written;
            }
            cv_free.notify_all();
            cv_done.notify_all();
        }
    }

    void convert_loop() {
        for (;;) {
            size_t idx;
            Item it;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_work.wait(lk, [&] { return stop || next_convert < pending.size(); });
                if (next_convert >= pending.size()) { if (stop) return; continue; }
                idx = next_convert++;
                it = pending[idx];
            }
            if (io.wait && io.wait(io.user, it.ticket) != 0) { std::lock_guard<std::mutex> lk(mu); error = POPPY_CUDA_ERR_CUDA; }
            if (io.convert) io.convert(io.user, it.frame_index, buffers[it.buffer], width, height, row_bytes);
            {
                std::lock_guard<std::mutex> lk(mu);
                // entries only leave at the front, and only after they are converted: find ours by frame index
                for (auto& p : pending)
                    if (p.frame_index == it.frame_index && p.buffer == it.buffer) { p.converted = true; break; }
            }
            cv_work.notify_all();
        }
    }
};

namespace {
int writer_create(poppy_host_writer** out, const poppy_host_writer_io* io, int width, int height, size_t row_bytes, size_t frame_bytes,
                  int ring_frames, int workers) {
    if (!out) return POPPY_CUDA_ERR_INVALID;
    *out = nullptr;
    if (!io || !io->download || !io->write || !io->alloc || !io->release || width <= 0 || height <= 0 || ring_frames < 1 || workers < 0)
        return POPPY_CUDA_ERR_INVALID;
    poppy_host_writer* w = new poppy_host_writer();
    w->io = *io;
    w->width = width; w->height = height; w->ring = ring_frames; w->workers = io->convert ? workers : 0;
    w->row_bytes = row_bytes; w->frame_bytes = frame_bytes;
    for (int i = 0; i < ring_frames; ++i) {
        void* p = nullptr;
        if (io->alloc(io->user, w->frame_bytes, &p) != 0 || !p) {
            for (uint8_t* b : w->buffers) io->release(io->user, b);
            delete w;
            return POPPY_CUDA_ERR_CUDA;
        }
        w->buffers.push_back((uint8_t*)p);
        w->free_buffers.push_back(i);
    }
    w->deliverer = std::thread([w] { w->deliver_loop(); });
    for (int i = 0; i < w->workers; ++i) w->pool.emplace_back([w] { w->convert_loop(); });
    *out = w;
    return 0;
}
}  // namespace

extern "C" {

int poppy_host_writer_create_io(poppy_host_writer** out, const poppy_host_writer_io* io, int width, int height, int ring_frames,
                                int workers) {
    return writer_create(out, io, width, height, (size_t)width * 3, (size_t)width * height * 3, ring_frames, workers);
}

int poppy_host_writer_submit(poppy_host_writer* w, int first_slot, int count, int first_frame_index) {
    if (!w || count < 0) return POPPY_CUDA_ERR_INVALID;
    for (int i = 0; i < count; ++i) {
        int buf;
        {
            std::unique_lock<std::mutex> lk(w->mu);
            w->cv_free.wait(lk, [&] { return !w->free_buffers.empty(); });       // back-pressure: the ring is full
            buf = w->free_buffers.front();
            w->free_buffers.pop_front();
        }
        uint64_t ticket = 0;
        const int rc = w->io.download(w->io.user, first_slot + i, w->buffers[buf], w->row_bytes, &ticket);
        if (rc != 0) {
            std::lock_guard<std::mutex> lk(w->mu);
            w->free_buffers.push_back(buf);
            return rc;
        }
        {
            std::lock_guard<std::mutex> lk(w->mu);
            w->pending.push_back({first_frame_index + i, buf, ticket, false});
            ++w->submitted;
        }
        w->cv_work.notify_all();
    }
    return 0;
}

int poppy_host_writer_flush(poppy_host_writer* w) {
    if (!w) return POPPY_CUDA_ERR_INVALID;
    std::unique_lock<std::mutex> lk(w->mu);
    w->cv_done.wait(lk, [&] { return w->written == w->submitted; });
    return w->error;
}

void poppy_host_writer_destroy(poppy_host_writer* w) {
    if (!w) return;
    poppy_host_writer_flush(w);
    {
        std::lock_guard<std::mutex> lk(w->mu);
        w->stop = true;
    }
    w->cv_work.notify_all();
    if (w->deliverer.joinable()) w->deliverer.join();
    for (auto& t : w->pool) t.join();
    for (uint8_t* b : w->buffers) w->io.release(w->io.user, b);
    delete w;
}

// ---- the CUDA transport: ring slots of a poppy_cuda context ---------------------------------------------------------------
namespace {
struct CudaTransport { poppy_cuda_ctx* ctx; poppy_write_fn write; poppy_write_fn convert; void* user; int w, h; };
int ct_download(void* u, int slot, uint8_t* dst, size_t step, uint64_t* ticket) {
    auto* t = (CudaTransport*)u;
    return poppy_cuda_download_async(t->ctx, slot, 1, dst, step, step * (size_t)t->h, ticket);
}
int ct_download_i420(void* u, int slot, uint8_t* dst, size_t, uint64_t* ticket) {
    auto* t = (CudaTransport*)u;
    return poppy_cuda_download_i420_async(t->ctx, slot, 1, dst, (size_t)t->w * t->h * 3 / 2, ticket);
}
int ct_wait(void* u, uint64_t ticket) { return poppy_cuda_download_wait(((CudaTransport*)u)->ctx, ticket); }
int ct_alloc(void*, size_t bytes, void** out) { return poppy_cuda_alloc_pinned(bytes, out); }
void ct_release(void*, void* p) { poppy_cuda_free_pinned(p); }
void ct_write(void* u, int idx, uint8_t* bgr, int w, int h, size_t step) { auto* t = (CudaTransport*)u; t->write(t->user, idx, bgr, w, h, step); }
void ct_convert(void* u, int idx, uint8_t* bgr, int w, int h, size_t step) { auto* t = (CudaTransport*)u; t->convert(t->user, idx, bgr, w, h, step); }

int cuda_writer_create(poppy_host_writer** out, poppy_cuda_ctx* ctx, int ring_frames, poppy_write_fn write, poppy_write_fn convert,
                       int workers, void* user, bool i420) {
    if (!out || !ctx || !write) return POPPY_CUDA_ERR_INVALID;
    int w = 0, h = 0;
    if (int rc = poppy_cuda_get_info(ctx, &w, &h, nullptr, nullptr, nullptr, nullptr)) return rc;
    if (i420 && ((w | h) & 1)) return POPPY_CUDA_ERR_INVALID;         // I420 needs an even frame size
    // at most 64 download tickets may be outstanding (poppy_cuda.h)
    if (ring_frames > 48) ring_frames = 48;
    auto* t = new CudaTransport{ctx, write, convert, user, w, h};
    poppy_host_writer_io io{};
    io.user = t; io.download = i420 ? ct_download_i420 : ct_download; io.wait = ct_wait; io.alloc = ct_alloc; io.release = ct_release;
    io.write = ct_write;
    io.convert = convert ? ct_convert : nullptr;
    const int rc = i420 ? writer_create(out, &io, w, h, (size_t)w, (size_t)w * h * 3 / 2, ring_frames, workers)
                        : poppy_host_writer_create_io(out, &io, w, h, ring_frames, workers);
    if (rc != 0) { delete t; return rc; }
    (*out)->io.owned_transport = t;
    return 0;
}
}  // namespace

int poppy_host_writer_create(poppy_host_writer** out, poppy_cuda_ctx* ctx, int ring_frames, poppy_write_fn write,
                             poppy_write_fn convert, int workers, void* user) {
    return cuda_writer_create(out, ctx, ring_frames, write, convert, workers, user, false);
}

int poppy_host_writer_create_i420(poppy_host_writer** out, poppy_cuda_ctx* ctx, int ring_frames, poppy_write_fn write,
                                  poppy_write_fn convert, int workers, void* user) {
    return cuda_writer_create(out, ctx, ring_frames, write, convert, workers, user, true);
}

namespace {

// FFV1: the ring buffers hold W*H*3 bytes + a margin, which every natural frame's packet fits. The encode is synchronous (the
// packet size is known only after it), so the transport has no wait step. A packet that does not fit its buffer (noise)
// goes to a heap buffer of its exact size, handed to `packet` in place of the ring buffer.
struct Ffv1Transport {
    poppy_cuda_ctx* ctx;
    poppy_packet_fn packet;
    void* user;
    size_t cap;
    std::mutex mu;
    std::map<const uint8_t*, std::vector<uint8_t>> large;   // ring buffer -> the packet that did not fit it
    std::map<const uint8_t*, size_t> size;                   // ring buffer -> its packet's size
};
int ft_download(void* u, int slot, uint8_t* dst, size_t, uint64_t* ticket) {
    auto* t = (Ffv1Transport*)u;
    uint32_t n = 0;
    *ticket = 0;
    int rc = poppy_cuda_download_ffv1(t->ctx, slot, 1, dst, t->cap, &n);
    if (rc == POPPY_CUDA_ERR_INVALID && n > t->cap) {
        std::vector<uint8_t> big(n);
        rc = poppy_cuda_download_ffv1(t->ctx, slot, 1, big.data(), big.size(), &n);
        if (rc == 0) { std::lock_guard<std::mutex> lk(t->mu); t->large[dst] = std::move(big); }
    }
    if (rc == 0) { std::lock_guard<std::mutex> lk(t->mu); t->size[dst] = n; }
    return rc;
}
void ft_write(void* u, int idx, uint8_t* buf, int, int, size_t) {
    auto* t = (Ffv1Transport*)u;
    std::vector<uint8_t> big;
    size_t n;
    {
        std::lock_guard<std::mutex> lk(t->mu);
        n = t->size[buf];
        auto it = t->large.find(buf);
        if (it != t->large.end()) { big = std::move(it->second); t->large.erase(it); }
    }
    t->packet(t->user, idx, big.empty() ? buf : big.data(), n);
}
}  // namespace

int poppy_host_writer_create_ffv1(poppy_host_writer** out, poppy_cuda_ctx* ctx, int ring_frames, poppy_packet_fn packet, void* user) {
    if (!out || !ctx || !packet) return POPPY_CUDA_ERR_INVALID;
    int w = 0, h = 0;
    if (int rc = poppy_cuda_get_info(ctx, &w, &h, nullptr, nullptr, nullptr, nullptr)) return rc;
    auto* t = new Ffv1Transport{ctx, packet, user, (size_t)w * h * 3 + 65536, {}, {}, {}};
    poppy_host_writer_io io{};
    io.user = t; io.download = ft_download; io.wait = nullptr; io.alloc = ct_alloc; io.release = ct_release; io.write = ft_write;
    const int rc = writer_create(out, &io, w, h, 0, t->cap, ring_frames, 0);
    if (rc != 0) { delete t; return rc; }
    (*out)->io.owned_transport = t;
    (*out)->owned_ffv1 = true;
    return 0;
}

void poppy_host_writer_destroy_cuda(poppy_host_writer* w) {
    if (!w) return;
    void* t = w->io.owned_transport;
    const bool ffv1 = w->owned_ffv1;
    poppy_host_writer_destroy(w);
    if (ffv1) delete (Ffv1Transport*)t;
    else delete (CudaTransport*)t;
}

}  // extern "C"
