// Input conditioning ahead of the morph path, once per image (SURVEY.md 8(f-3)): poppy::blur_margin
// (reference src/util.cpp:574-602) on the GPU - the source centred on a black union-sized canvas whose left, right, top
// and bottom margins are blurred by an 8-bit cv::GaussianBlur(127 x 127, sigma 6), all four from the unblurred canvas and
// written in that order.
//
// OpenCV 4.6.0 evaluates an 8-bit GaussianBlur of an isolated image in fixed point
// (OCV imgproc/src/smooth.dispatch.cpp:654-684): taps = the bit-exact Gaussian scaled to 8 fractional bits with error
// diffusion (:82-198, :224-259); rows h = sum m[k] * src[reflect101] in 16 bits (smooth.simd.hpp:1136-1199); columns
// v = sum m[k] * h[reflect101] in 32 bits, out = (v + 2^15) >> 16 (:1780-1866). Integer sums: order is immaterial and
// nothing can overflow (the taps add up to 256), so the kernels below are exact by construction; of the 127 taps only
// the 35 central ones are non-zero at sigma 6.
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/poppy_cuda.h"
#include "device/kernels.cuh"
#include "device/pixel_ops.cuh"

namespace poppy {
namespace {

constexpr int MG_KSIZE = 127;
constexpr double MG_SIGMA = 6.0;
__constant__ int c_margin_taps[MG_KSIZE];

// getGaussianKernelBitExact + getGaussianKernelFixedPoint_ED (softdouble = IEEE double operations, round half to even)
std::vector<int> gaussian_kernel_fixed(int n, double sigma, int bits) {
    const double scale2x = -0.125 / (sigma * sigma);
    const int n2 = (n - 1) / 2;
    std::vector<double> vals(n2);
    double sum = 0.0;
    for (int i = 0, x = 1 - n; i < n2; ++i, x += 2) {
        vals[i] = std::exp((double)(x * x) * scale2x);
        sum += vals[i];
    }
    sum *= 2.0;
    sum += 1.0;
    const double mul1 = 1.0 / sum;
    std::vector<int> res(n, 0);
    double err = 0.0;
    long long total = 0;
    for (int i = 0; i < n2; ++i) {
        const double adj = vals[i] * mul1 * (double)(1ll << bits) + err;
        const long long v0 = std::llrint(adj);
        err = adj - (double)v0;
        res[i] = res[n - 1 - i] = (int)v0;
        total += v0;
    }
    res[n2] = (int)((1ll << bits) - 2 * total);
    return res;
}

__device__ __forceinline__ int margin_reflect(int p, int len) {      // cv::borderInterpolate, BORDER_REFLECT_101
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * (len - 1) - p;
    return p;
}

// rows of one margin rectangle: tmp[y][x * 3 + c] = sum_k taps[k] * canvas(x0 + reflect(x + k - r), y0 + y, c)
// grid (ceil(3 w / 256), h); k_lo .. k_hi: the non-zero taps; one_px: the axis is one pixel long (kernel shrinks to [1])
__global__ void k_margin_rows(const uint8_t* __restrict__ canvas, size_t pitch, int x0, int y0, int w, int h, int k_lo, int k_hi,
                              int one_px, uint16_t* __restrict__ tmp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (i >= 3 * w) return;
    const int x = i / 3, c = i - 3 * x;
    const uint8_t* __restrict__ row = canvas + (size_t)(y0 + y) * pitch + (size_t)x0 * 3 + c;
    unsigned acc = 0;
    if (one_px) {
        acc = 256u * row[0];
    } else {
        for (int k = k_lo; k <= k_hi; ++k) acc += (unsigned)c_margin_taps[k] * row[3 * margin_reflect(x + k - MG_KSIZE / 2, w)];
    }
    tmp[(size_t)y * 3 * w + i] = (uint16_t)acc;
}

// columns: out(x0 + x, y0 + y, c) = min(255, (sum_k taps[k] * tmp[reflect(y + k - r)][x * 3 + c] + 2^15) >> 16)
__global__ void k_margin_cols(const uint16_t* __restrict__ tmp, int x0, int y0, int w, int h, int k_lo, int k_hi, int one_px,
                              uint8_t* __restrict__ out, size_t pitch) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (i >= 3 * w) return;
    unsigned acc = 0;
    if (one_px) {
        acc = 256u * tmp[(size_t)y * 3 * w + i];
    } else {
        for (int k = k_lo; k <= k_hi; ++k) acc += (unsigned)c_margin_taps[k] * tmp[(size_t)margin_reflect(y + k - MG_KSIZE / 2, h) * 3 * w + i];
    }
    const unsigned v = (acc + (1u << 15)) >> 16;
    out[(size_t)(y0 + y) * pitch + (size_t)x0 * 3 + i] = (uint8_t)(v > 255u ? 255u : v);
}

// ---- gabor_filter (reference src/util.cpp:40-60, defaults as src/poppy.hpp:122 calls it) ----------------------------------------
// dst = (1/16) sum_i clamp01(filter2D(src, gaborKernel_i)); cv::filter2D sends a 13 x 13 float kernel over a float image
// through crossCorr, which promotes to DOUBLE, correlates by block DFT and rounds back to float (filter.dispatch.cpp:1291,
// templmatch.cpp:592). Here the same correlation is summed directly in double (BORDER_REFLECT_101, centre anchor): equal
// to the DFT evaluation to ~1e-15, so the float results differ only where the exact value sits on a float rounding
// boundary (measured: 0-1 values per million, by one ulp). Floating-point parity with a stated tolerance, not bit-exact.
constexpr int GB_ANGLES = 16, GB_K = 13, GB_R = GB_K / 2, GB_TW = 32, GB_TH = 4, GB_TW3 = (GB_TW + 2 * GB_R) * 3;
__constant__ double c_gabor_taps[GB_ANGLES * GB_K * GB_K];

// a source value as the filter sees it: a float image as given, an 8-bit one as convertTo(CV_32F, 1/255) makes it -
// float(v) * float(1/255.0), one rounding (OCV core/src/convert_scale.simd.hpp:91-125); not v / 255
__device__ __forceinline__ float gabor_in(float v) { return v; }
__device__ __forceinline__ float gabor_in(uint8_t v) { return __fmul_rn((float)v, kInv255); }

// the block's 32 x 4 pixels with a 6-pixel apron (BORDER_REFLECT_101), channels interleaved: tile[row][x * 3 + c]
template <class T>
__device__ __forceinline__ void gabor_load_tile(float (*tile)[GB_TW3], const T* __restrict__ src, size_t spitch, int w, int h) {
    const int bx = blockIdx.x * GB_TW, by = blockIdx.y * GB_TH;
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    for (int i = tid; i < (GB_TH + 2 * GB_R) * GB_TW3; i += 3 * GB_TW * GB_TH) {
        const int ty = i / GB_TW3, tx = i - ty * GB_TW3, px = tx / 3, c = tx - 3 * px;
        const int gx = margin_reflect(bx + px - GB_R, w), gy = margin_reflect(by + ty - GB_R, h);
        tile[ty][tx] = gabor_in(src[(size_t)gy * spitch + (size_t)gx * 3 + c]);
    }
}

// dst(x, y, c) for the pixel at tile column px of tile row `row`
__device__ __forceinline__ float gabor_value(const float (*tile)[GB_TW3], int row, int px, int c) {
    double acc[GB_ANGLES];
#pragma unroll
    for (int a = 0; a < GB_ANGLES; ++a) acc[a] = 0.0;
#pragma unroll 1
    for (int i = 0; i < GB_K; ++i) {
#pragma unroll
        for (int j = 0; j < GB_K; ++j) {
            const double v = (double)tile[row + i][(px + j) * 3 + c];
#pragma unroll
            for (int a = 0; a < GB_ANGLES; ++a) acc[a] = fma(c_gabor_taps[(a * GB_K + i) * GB_K + j], v, acc[a]);
        }
    }
    float sum = 0.f;
#pragma unroll
    for (int a = 0; a < GB_ANGLES; ++a) {
        float p = (float)acc[a];                 // crossCorr converts its double result to the float plane
        p = p > 1.f ? 1.f : p;                   // plane.setTo(1, plane > 1); plane.setTo(0, plane < 0)
        p = p < 0.f ? 0.f : p;
        sum = __fadd_rn(sum, p);                 // dst += plane
    }
    return __fmul_rn(sum, 1.f / GB_ANGLES);      // dst /= 16
}

// block (96, 4): thread = (pixel x within the 32-pixel tile, channel) x row; grid (ceil(w / 32), ceil(h / 4))
__global__ void __launch_bounds__(3 * GB_TW * GB_TH)
k_gabor(const float* __restrict__ src, size_t spitch, int w, int h, float* __restrict__ dst, size_t dpitch) {
    __shared__ float tile[GB_TH + 2 * GB_R][GB_TW3];
    gabor_load_tile(tile, src, spitch, w, h);
    __syncthreads();
    const int px = threadIdx.x / 3, c = threadIdx.x - 3 * px, gx = blockIdx.x * GB_TW + px, gy = blockIdx.y * GB_TH + threadIdx.y;
    if (gx >= w || gy >= h) return;
    dst[(size_t)gy * dpitch + (size_t)gx * 3 + c] = gabor_value(tile, threadIdx.y, px, c);
}

// The mask basis straight from the 8-bit corrected2 (tight rows): m2 = 1 - gray(gabor_filter(corrected2 * 1/255)), the
// gabor2 of reference src/poppy.hpp:119-122 reduced as src/algo.cpp:250-252 reduces it, without gabor2 ever being stored.
// Same block shape and arithmetic as k_gabor. The three channels of a pixel come from threads 3 px .. 3 px + 2, which may
// sit in two warps, so they meet in shared memory; then thread px of each row finishes pixel px.
__global__ void __launch_bounds__(3 * GB_TW * GB_TH)
k_gabor_mask_basis(const uint8_t* __restrict__ src, int w, int h, float* __restrict__ m2, int bpitch) {
    __shared__ float tile[GB_TH + 2 * GB_R][GB_TW3];
    __shared__ float gab[GB_TH][3 * GB_TW];
    gabor_load_tile(tile, src, (size_t)w * 3, w, h);
    __syncthreads();
    const int bx = blockIdx.x * GB_TW, px = threadIdx.x / 3, c = threadIdx.x - 3 * px, gy = blockIdx.y * GB_TH + threadIdx.y;
    if (bx + px < w && gy < h) gab[threadIdx.y][threadIdx.x] = gabor_value(tile, threadIdx.y, px, c);
    __syncthreads();
    const int x = bx + threadIdx.x;
    if (threadIdx.x >= GB_TW || x >= w || gy >= h) return;
    const float* g = gab[threadIdx.y] + 3 * threadIdx.x;
    m2[(size_t)gy * bpitch + x] = mask_basis_px(g[0], g[1], g[2], x < (w & ~7));
}

// cv::getGaborKernel(Size(13, 13), sigma, theta, lambda, gamma, psi, CV_32F) (OCV imgproc/src/gabor.cpp:51-95)
void gabor_kernel(double sigma, double theta, double lambd, double gamma, double psi, float* k) {
    const double sigma_x = sigma, sigma_y = sigma / gamma, c = std::cos(theta), s = std::sin(theta);
    const double ex = -0.5 / (sigma_x * sigma_x), ey = -0.5 / (sigma_y * sigma_y), cscale = 3.1415926535897932384626433832795 * 2 / lambd;
    for (int y = -GB_R; y <= GB_R; ++y)
        for (int x = -GB_R; x <= GB_R; ++x) {
            const double xr = x * c + y * s, yr = -x * s + y * c;
            const double v = 1.0 * std::exp(ex * xr * xr + ey * yr * yr) * std::cos(cscale * xr + psi);
            k[(GB_R - y) * GB_K + (GB_R - x)] = (float)v;
        }
}

// the 16 kernels as c_gabor_taps holds them: theta_i = i * float(180 / 16) - an integer division, and degrees where radians
// are expected, as in the reference (src/util.cpp:43-46); sigma 5, lambda 10, gamma 0.04, psi pi/4 (src/util.hpp:95)
const std::vector<double>& gabor_taps() {
    static const std::vector<double> taps = [] {
        std::vector<double> t((size_t)GB_ANGLES * GB_K * GB_K);
        const float step = (float)(180 / GB_ANGLES);
        for (int a = 0; a < GB_ANGLES; ++a) {
            float k[GB_K * GB_K];
            gabor_kernel(5.0, (double)(a * step), 10.0, 0.04, 3.1415926535897932384626433832795 / 4, k);
            for (int i = 0; i < GB_K * GB_K; ++i) t[(size_t)a * GB_K * GB_K + i] = (double)k[i];
        }
        return t;
    }();
    return taps;
}

thread_local std::string g_margin_error;
int margin_fail(int code, const std::string& msg) {
    g_margin_error = msg;
    return code;
}

struct Rect { int x, y, w, h; };

}  // namespace

void margin_set_error(const std::string& msg) { g_margin_error = msg; }

cudaError_t launch_gabor_mask_basis(cudaStream_t st, const uint8_t* bgr, float* m2, int bpitch, int w, int h) {
    // c_gabor_taps: written once per device. The copy is complete before the flag is raised, so a context on another stream
    // of the same device never launches ahead of it (poppy_cuda_gabor_filter rewrites the same values).
    static std::atomic<bool> taps_ready[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const bool tracked = dev >= 0 && dev < 64;
    if (!tracked || !taps_ready[dev].load(std::memory_order_acquire)) {
        const std::vector<double>& taps = gabor_taps();
        e = cudaMemcpyToSymbolAsync(c_gabor_taps, taps.data(), taps.size() * sizeof(double), 0, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return e;
        if (tracked) taps_ready[dev].store(true, std::memory_order_release);
    }
    k_gabor_mask_basis<<<dim3(div_up(w, GB_TW), div_up(h, GB_TH)), dim3(3 * GB_TW, GB_TH), 0, st>>>(bgr, w, h, m2, bpitch);
    return cudaGetLastError();
}

}  // namespace poppy

extern "C" {

const char* poppy_cuda_blur_margin_last_error(void) { return poppy::g_margin_error.c_str(); }

int poppy_cuda_blur_margin(int device, const uint8_t* src, size_t src_step, int cols, int rows, int union_w, int union_h,
                           uint8_t* dst, size_t dst_step) {
    using namespace poppy;
    if (!src || !dst || cols < 1 || rows < 1 || union_w < 1 || union_h < 1 || src_step < (size_t)cols * 3 || dst_step < (size_t)union_w * 3)
        return margin_fail(POPPY_CUDA_ERR_INVALID, "blur_margin: bad argument");
    // the geometry of src/util.cpp:577-592 with its double -> int truncations; cv::Mat::operator()(Rect) throws where a
    // rectangle leaves the canvas
    const double margin_factor = 1.3, margin = (cols + rows) / 100.0;
    double dx = std::fabs((double)cols - union_w) / 2.0, dy = std::fabs((double)rows - union_h) / 2.0;
    const Rect roi{(int)dx, (int)dy, cols, rows};
    dx = dx == 0 ? margin_factor : dx + margin;
    dy = dy == 0 ? margin_factor : dy + margin;
    const Rect rects[4] = {{0, 0, (int)dx, union_h}, {(int)(union_w - dx), 0, (int)dx, union_h},
                           {0, 0, union_w, (int)dy}, {0, (int)(union_h - dy), union_w, (int)dy}};
    auto inside = [&](const Rect& r) { return r.x >= 0 && r.y >= 0 && r.w >= 1 && r.h >= 1 && r.x + r.w <= union_w && r.y + r.h <= union_h; };
    if (!inside(roi)) return margin_fail(POPPY_CUDA_ERR_INVALID, "blur_margin: the source does not fit the union size (cv::Mat ROI assertion)");
    for (const Rect& r : rects)
        if (!inside(r)) return margin_fail(POPPY_CUDA_ERR_INVALID, "blur_margin: a margin rectangle leaves the canvas (cv::Mat ROI assertion)");

    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev < 1 || device < 0 || device >= n_dev)
        return margin_fail(POPPY_CUDA_ERR_NO_DEVICE, "blur_margin: no such CUDA device (there is no CPU fallback)");
#define MG_TRY(expr)                                                                                                  \
    do {                                                                                                              \
        cudaError_t e_ = (expr);                                                                                      \
        if (e_ != cudaSuccess) {                                                                                      \
            cudaFree(d_canvas); cudaFree(d_out); cudaFree(d_tmp);                                                     \
            return margin_fail(POPPY_CUDA_ERR_CUDA, std::string("blur_margin: ") + cudaGetErrorString(e_));           \
        }                                                                                                             \
    } while (0)
    uint8_t *d_canvas = nullptr, *d_out = nullptr;
    uint16_t* d_tmp = nullptr;
    MG_TRY(cudaSetDevice(device));
    const std::vector<int> taps = gaussian_kernel_fixed(MG_KSIZE, MG_SIGMA, 8);
    int k_lo = 0, k_hi = MG_KSIZE - 1;
    while (k_lo < MG_KSIZE / 2 && taps[k_lo] == 0) ++k_lo;
    while (k_hi > MG_KSIZE / 2 && taps[k_hi] == 0) --k_hi;
    MG_TRY(cudaMemcpyToSymbol(c_margin_taps, taps.data(), sizeof(int) * MG_KSIZE));
    const size_t pitch = (size_t)union_w * 3, bytes = pitch * union_h;
    size_t tmp_elems = 0;
    for (const Rect& r : rects) tmp_elems = std::max(tmp_elems, (size_t)r.w * r.h * 3);
    MG_TRY(cudaMalloc((void**)&d_canvas, bytes));
    MG_TRY(cudaMalloc((void**)&d_out, bytes));
    MG_TRY(cudaMalloc((void**)&d_tmp, tmp_elems * sizeof(uint16_t)));
    MG_TRY(cudaMemset(d_canvas, 0, bytes));
    MG_TRY(cudaMemcpy2D(d_canvas + (size_t)roi.y * pitch + (size_t)roi.x * 3, pitch, src, src_step, (size_t)cols * 3, rows,
                        cudaMemcpyHostToDevice));
    MG_TRY(cudaMemcpy(d_out, d_canvas, bytes, cudaMemcpyDeviceToDevice));
    for (const Rect& r : rects) {
        const dim3 grid(div_up(3 * r.w, 256), r.h);
        k_margin_rows<<<grid, 256>>>(d_canvas, pitch, r.x, r.y, r.w, r.h, k_lo, k_hi, r.w == 1, d_tmp);
        k_margin_cols<<<grid, 256>>>(d_tmp, r.x, r.y, r.w, r.h, k_lo, k_hi, r.h == 1, d_out, pitch);
    }
    MG_TRY(cudaGetLastError());
    MG_TRY(cudaMemcpy2D(dst, dst_step, d_out, pitch, pitch, union_h, cudaMemcpyDeviceToHost));
#undef MG_TRY
    cudaFree(d_canvas); cudaFree(d_out); cudaFree(d_tmp);
    return 0;
}

int poppy_cuda_gabor_filter(int device, const float* src, size_t src_step, int cols, int rows, float* dst, size_t dst_step) {
    using namespace poppy;
    if (!src || !dst || cols < 1 || rows < 1 || src_step < (size_t)cols * 12 || dst_step < (size_t)cols * 12 || src_step % 4 || dst_step % 4)
        return margin_fail(POPPY_CUDA_ERR_INVALID, "gabor_filter: bad argument");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev < 1 || device < 0 || device >= n_dev)
        return margin_fail(POPPY_CUDA_ERR_NO_DEVICE, "gabor_filter: no such CUDA device (there is no CPU fallback)");
    float *d_src = nullptr, *d_dst = nullptr;
#define GB_TRY(expr)                                                                                                  \
    do {                                                                                                              \
        cudaError_t e_ = (expr);                                                                                      \
        if (e_ != cudaSuccess) {                                                                                      \
            cudaFree(d_src); cudaFree(d_dst);                                                                         \
            return margin_fail(POPPY_CUDA_ERR_CUDA, std::string("gabor_filter: ") + cudaGetErrorString(e_));          \
        }                                                                                                             \
    } while (0)
    GB_TRY(cudaSetDevice(device));
    const std::vector<double>& taps = gabor_taps();
    GB_TRY(cudaMemcpyToSymbol(c_gabor_taps, taps.data(), taps.size() * sizeof(double)));
    const size_t pitch = (size_t)cols * 3;
    GB_TRY(cudaMalloc((void**)&d_src, pitch * rows * sizeof(float)));
    GB_TRY(cudaMalloc((void**)&d_dst, pitch * rows * sizeof(float)));
    GB_TRY(cudaMemcpy2D(d_src, pitch * 4, src, src_step, pitch * 4, rows, cudaMemcpyHostToDevice));
    k_gabor<<<dim3(div_up(cols, GB_TW), div_up(rows, GB_TH)), dim3(3 * GB_TW, GB_TH)>>>(d_src, pitch, cols, rows, d_dst, pitch);
    GB_TRY(cudaGetLastError());
    GB_TRY(cudaMemcpy2D(dst, dst_step, d_dst, pitch * 4, pitch * 4, rows, cudaMemcpyDeviceToHost));
#undef GB_TRY
    cudaFree(d_src); cudaFree(d_dst);
    return 0;
}

}  // extern "C"
