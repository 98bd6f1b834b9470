// C++ host shim with the reference's interface for the morph path: poppy::Settings (reference src/settings.hpp:9-35)
// and poppy::morph_images() (reference src/algo.hpp:26). Argument order, meaning, by-value point vectors, the
// morphedPoints out-parameter and the "returns 0" convention are the reference's; images are passed as light views
// instead of cv::Mat so that this header has no OpenCV dependency (include/poppy_morph_cv.hpp adapts cv::Mat).
//
// Host stages (clip/uniq/Delaunay/index lookup) run here; everything from morph_points() to the 8-bit frame runs on
// the GPU through include/poppy_cuda.h. There is no CPU rendering path: without a CUDA device morph_images throws.
#pragma once

#include <cstddef>
#include <cstdint>
#include <functional>
#include <stdexcept>
#include <string>
#include <vector>

#include "delaunay.hpp"

namespace poppy {

class Settings {
    static Settings* instance_;
    Settings() {}

public:
    bool show_gui = false;
    bool enable_wait = false;
    double number_of_frames = 60;
    double frame_rate = 30;
    double match_tolerance = 1;
    size_t max_keypoints = 300;
    size_t pyramid_levels = 64;
    bool enable_auto_align = false;
    bool enable_radial_mask = false;
    bool enable_face_detection = false;
    bool enable_denoise = false;
    bool enable_src_scaling = false;
    size_t face_neighbors = 8;
    std::string fourcc = "FFV1";
    int cuda_device = 0;               // addition: which GPU the renderer uses

    static Settings& instance() {
        if (instance_ == nullptr) instance_ = new Settings();
        return *instance_;
    }
};

// 8UC3 (BGR) image view / owner. `data` may point into a cv::Mat.
struct Image8 {
    uint8_t* data = nullptr;
    int cols = 0, rows = 0;
    size_t step = 0;
    std::vector<uint8_t> owned;
    bool empty() const { return data == nullptr || cols == 0 || rows == 0; }
    void create(int c, int r) {
        cols = c; rows = r; step = (size_t)c * 3;
        owned.assign(step * r, 0);
        data = owned.data();
    }
};

// 32FC3 image view (gabor2)
struct Image32F {
    const float* data = nullptr;
    int cols = 0, rows = 0;
    size_t step = 0;   // bytes
};

class MorphError : public std::runtime_error {
public:
    using std::runtime_error::runtime_error;
};
// thrown by calls that check for a CUDA device up front when the machine has none
class NoDeviceError : public MorphError {
public:
    using MorphError::MorphError;
};

// reference src/algo.hpp:26 / src/algo.cpp:178-273. img1 supplies only the frame size; goodFeatures1/2, img2, last
// and linear are unused exactly as in the reference. dst is (re)allocated when its size differs.
double morph_images(const Image8& img1, const Image8& img2, const Image8& corrected1, const Image8& corrected2,
                    const Image32F& gabor2, Image8& goodFeatures1, Image8& goodFeatures2, Image8& dst,
                    const Image8& last, std::vector<Point2f>& morphedPoints, std::vector<Point2f> srcPoints1,
                    std::vector<Point2f> srcPoints2, double shapeRatio, double maskRatio, double linear);

// The frame loop of morph<Twriter>() (reference src/poppy.hpp:177-243, phase < 0) with the whole segment resident
// on the GPU: points/topology of all frames are planned on host threads, the chain is rendered with frame j-1 kept
// in HBM as frame j's source, and frames are handed to `write` in order. An empty gabor2 (data == nullptr) has the
// device derive it from corrected2, as poppy::morph() does before its frame loop (src/poppy.hpp:119-122).
void morph_sequence(const Image8& corrected1, const Image8& corrected2, const Image32F& gabor2,
                    std::vector<Point2f> srcPoints1, std::vector<Point2f> srcPoints2, int number_of_frames,
                    const std::function<void(const Image8&)>& write);
// The same with gabor2 derived on the device from corrected2: only the two 8-bit images cross PCIe.
void morph_sequence(const Image8& corrected1, const Image8& corrected2, std::vector<Point2f> srcPoints1,
                    std::vector<Point2f> srcPoints2, int number_of_frames, const std::function<void(const Image8&)>& write);

// One segment of a multi-image sequence: the arguments of morph_sequence for one consecutive pair.
struct Segment {
    Image8 corrected1, corrected2;
    Image32F gabor2;                   // empty: derived on the device
    std::vector<Point2f> srcPoints1, srcPoints2;
};
// The segments of run() (reference src/poppy.cpp:266-328), each the chain morph_sequence renders, rendered together on the
// GPU (step j of a group of segments per kernel batch). Frames go to `write` in the reference's order: all
// number_of_frames frames of segment 0, then segment 1, ...; segment 0's are written while later steps still render.
void morph_segments(const std::vector<Segment>& segments, int number_of_frames, const std::function<void(const Image8&)>& write);
// The same on several GPUs of one box: the K segments are sharded over the first G = min(devices.size(), K) listed devices,
// devices[g] rendering the contiguous range [g * K / G, (g + 1) * K / G) on its own context and host thread; the other
// listed devices stay idle. The frames and the order of the `write` calls equal the single-device call's: `write` is
// called from a library thread, one call at a time. The device list is checked before anything is planned or rendered:
// MorphError for an empty list, a duplicate, a negative index or an index >= the device count, NoDeviceError without a GPU.
// If one device fails, the others stop at their next render call and the first error is thrown once all have stopped.
void morph_segments(const std::vector<Segment>& segments, int number_of_frames, const std::function<void(const Image8&)>& write,
                    const std::vector<int>& devices);

// Releases the cached device contexts (one per device) held by morph_images()/morph_sequence()/morph_segments().
void release_cached_contexts();

}  // namespace poppy
