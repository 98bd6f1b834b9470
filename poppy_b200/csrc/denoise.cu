// cv::fastNlMeansDenoising(src, dst, h, templateWindowSize, searchWindowSize) of an 8-bit BGR image on the GPU, as the
// reference's run() calls it under --denoise (src/poppy.cpp:172 for the first image, 269-311 for the later ones).
//
// OpenCV runs FastNlMeansDenoisingInvoker<Vec3b, int, unsigned, DistSquared, int> (photo/src/fast_nlmeans_denoising_invoker.hpp):
//   th = tw / 2, sh = sw / 2 (even sizes round up to 2 th + 1, 2 sh + 1); the source extended by sh + th on every side
//   (BORDER_REFLECT_101); for every pixel p and every offset o of the search window (o = 0 included)
//     D(p, o) = sum over the template around p of sum_c (I(q) - I(q + o))^2        (exact, int)
//     wt = lut[D >> shift];  W += wt;  E_c += wt * I_c(p + o)
//   out_c = saturate_u8((unsigned)(E_c + W / 2) / (unsigned)W).
// The weight table is the only floating-point step; it is built on the host with std::exp exactly as OpenCV builds it
// (denoise_weights below). Everything per pixel is integer arithmetic that cannot overflow (W <= sw^2 * mult <= INT_MAX / 255,
// E_c <= 255 W), so the order of summation is immaterial and any tiling gives OpenCV's bytes.
#include <algorithm>
#include <cmath>
#include <climits>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/poppy_cuda.h"
#include "device/common.cuh"

namespace poppy {

void margin_set_error(const std::string& msg);     // margin.cu: the per-thread text of poppy_cuda_blur_margin_last_error

namespace {

constexpr int NL_TX = 32;                // output tile: 32 columns (a warp's lanes) x 64 rows; 8 warps of 8 rows each
constexpr int NL_TY = 64;
constexpr int NL_RY = NL_TY / 8;         // rows per thread in the vertical pass
constexpr int NL_RX = 16;                // columns per thread in the horizontal pass
constexpr int NL_THREADS = 256;
constexpr int NL_HP = NL_TX + 1;         // row pitch (words) of the horizontal sums: odd, so both passes are conflict-free
constexpr int NL_MAX_TH = 7;             // template_window_size <= 15 after rounding
constexpr int NL_MAX_SH = 31;            // search_window_size <= 63 after rounding

// OpenCV's DistSquared for Vec3b, on BGRX words with X = 0: per-byte |a - b|, then the dot product of that with itself
__device__ __forceinline__ int sq_dist(uint32_t a, uint32_t b) {
    const uint32_t v = __vabsdiffu4(a, b);
    return (int)__dp4a(v, v, 0u);
}

__device__ __forceinline__ int nl_reflect(int p, int len) {      // cv::borderInterpolate, BORDER_REFLECT_101
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * (len - 1) - p;
    return p;
}

// One 32 x 64 tile of outputs per CTA. Shared memory: the extended source of the tile (border B = sh + TH) as BGRX words,
// two buffers of horizontal template sums, and (SMEM_LUT) the weight table's non-zero prefix plus one 0.
// Per offset o: pass 1 - thread t < (64 + 2 TH) * 2 owns row t / 2 (tile rows -TH .. 63 + TH) and 16 columns, and writes
// Hs(x, y) = sum_{|j| <= TH} d(x + j, y) by a running sum; pass 2 - lane x of warp g takes D(x, y) = sum_{|i| <= TH} Hs(x, y + i)
// for rows 8 g .. 8 g + 7 by a running sum and accumulates the weights. Double-buffered sums: one barrier per offset.
// lut_n: index of the table's first zero (the clamp; every later entry is 0 too, since the weights fall with D).
template <int TH, bool SMEM_LUT>
__global__ void __launch_bounds__(NL_THREADS, 3)
k_denoise(const uint8_t* __restrict__ src, int cols, int rows, int sh, const int* __restrict__ lut, int lut_n, int shift,
          uint8_t* __restrict__ dst) {
    extern __shared__ uint32_t nl_smem[];
    const int B = sh + TH, SP = NL_TX + 2 * B + 1, SR = NL_TY + 2 * B;     // SP odd: conflict-free pass-1 reads
    uint32_t* S = nl_smem;
    int* Hs = (int*)(S + SR * SP);
    constexpr int HR = NL_TY + 2 * TH, HWORDS = HR * NL_HP;
    const int* tab = lut;
    if constexpr (SMEM_LUT) {
        int* s_lut = Hs + 2 * HWORDS;
        for (int i = threadIdx.x; i <= lut_n; i += NL_THREADS) s_lut[i] = lut[i];
        tab = s_lut;
    }
    const int x0 = blockIdx.x * NL_TX, y0 = blockIdx.y * NL_TY, tid = threadIdx.x;
    for (int i = tid; i < SR * (NL_TX + 2 * B); i += NL_THREADS) {
        const int ty = i / (NL_TX + 2 * B), tx = i - ty * (NL_TX + 2 * B);
        const uint8_t* p = src + ((size_t)nl_reflect(y0 - B + ty, rows) * cols + nl_reflect(x0 - B + tx, cols)) * 3;
        S[ty * SP + tx] = (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16;
    }
    __syncthreads();

    // pass 1 ownership
    constexpr int NR = NL_RX + 2 * TH;
    const bool p1 = tid < HR * (NL_TX / NL_RX);
    const int r1 = tid / (NL_TX / NL_RX), c1 = (tid % (NL_TX / NL_RX)) * NL_RX;
    const uint32_t* cen = S + (r1 - TH + B) * SP + (c1 - TH + B);      // the first template centre of the run

    // pass 2 ownership
    const int lane = tid & 31, r2 = (tid >> 5) * NL_RY;
    unsigned W[NL_RY], E0[NL_RY], E1[NL_RY], E2[NL_RY];
#pragma unroll
    for (int j = 0; j < NL_RY; ++j) W[j] = E0[j] = E1[j] = E2[j] = 0u;

    int buf = 0;
    for (int dy = -sh; dy <= sh; ++dy) {
        for (int dx = -sh; dx <= sh; ++dx, buf ^= 1) {
            int* H = Hs + buf * HWORDS;
            if (p1) {
                const uint32_t* nb = cen + dy * SP + dx;
                int d[NR];
#pragma unroll
                for (int i = 0; i < NR; ++i) d[i] = sq_dist(cen[i], nb[i]);
                int s = 0;
#pragma unroll
                for (int i = 0; i <= 2 * TH; ++i) s += d[i];
                int* hrow = H + r1 * NL_HP + c1;
                hrow[0] = s;
#pragma unroll
                for (int j = 1; j < NL_RX; ++j) {
                    s += d[j + 2 * TH] - d[j - 1];
                    hrow[j] = s;
                }
            }
            __syncthreads();
            int hv[NL_RY + 2 * TH];
#pragma unroll
            for (int k = 0; k < NL_RY + 2 * TH; ++k) hv[k] = H[(r2 + k) * NL_HP + lane];
            const uint32_t* px = S + (r2 + B + dy) * SP + lane + B + dx;
            int D = 0;
#pragma unroll
            for (int i = 0; i <= 2 * TH; ++i) D += hv[i];
#pragma unroll
            for (int j = 0; j < NL_RY; ++j) {
                if (j) D += hv[j + 2 * TH] - hv[j - 1];
                const unsigned wt = (unsigned)tab[min(D >> shift, lut_n)];
                const uint32_t v = px[j * SP];
                W[j] += wt;
                E0[j] += wt * (v & 0xffu);
                E1[j] += wt * ((v >> 8) & 0xffu);
                E2[j] += wt * (v >> 16);
            }
        }
    }

    const int x = x0 + lane;
    if (x >= cols) return;
#pragma unroll
    for (int j = 0; j < NL_RY; ++j) {
        const int y = y0 + r2 + j;
        if (y >= rows) break;
        uint8_t* o = dst + ((size_t)y * cols + x) * 3;
        const unsigned half = W[j] / 2u;                     // E_c <= 255 W, so no quotient exceeds 255
        o[0] = (uint8_t)((E0[j] + half) / W[j]);
        o[1] = (uint8_t)((E1[j] + half) / W[j]);
        o[2] = (uint8_t)((E2[j] + half) / W[j]);
    }
}

size_t denoise_smem_bytes(int th, int sh, size_t lut_words) {
    const int B = sh + th;
    return sizeof(uint32_t) * ((size_t)(NL_TY + 2 * B) * (NL_TX + 2 * B + 1) + 2 * (size_t)(NL_TY + 2 * th) * NL_HP + lut_words);
}

template <int TH, bool SMEM_LUT>
cudaError_t launch_denoise_t(const uint8_t* src, int cols, int rows, int sh, const int* lut, int lut_n, int shift, uint8_t* dst,
                             size_t smem) {
    cudaError_t e = cudaFuncSetAttribute(k_denoise<TH, SMEM_LUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_denoise<TH, SMEM_LUT><<<dim3(div_up(cols, NL_TX), div_up(rows, NL_TY)), NL_THREADS, smem>>>(src, cols, rows, sh, lut, lut_n,
                                                                                                   shift, dst);
    return cudaGetLastError();
}

template <bool SMEM_LUT>
cudaError_t launch_denoise(int th, const uint8_t* src, int cols, int rows, int sh, const int* lut, int lut_n, int shift, uint8_t* dst,
                           size_t smem) {
    switch (th) {
        case 0: return launch_denoise_t<0, SMEM_LUT>(src, cols, rows, sh, lut, lut_n, shift, dst, smem);
        case 1: return launch_denoise_t<1, SMEM_LUT>(src, cols, rows, sh, lut, lut_n, shift, dst, smem);
        case 2: return launch_denoise_t<2, SMEM_LUT>(src, cols, rows, sh, lut, lut_n, shift, dst, smem);
        case 3: return launch_denoise_t<3, SMEM_LUT>(src, cols, rows, sh, lut, lut_n, shift, dst, smem);
        case 4: return launch_denoise_t<4, SMEM_LUT>(src, cols, rows, sh, lut, lut_n, shift, dst, smem);
        case 5: return launch_denoise_t<5, SMEM_LUT>(src, cols, rows, sh, lut, lut_n, shift, dst, smem);
        case 6: return launch_denoise_t<6, SMEM_LUT>(src, cols, rows, sh, lut, lut_n, shift, dst, smem);
        default: return launch_denoise_t<7, SMEM_LUT>(src, cols, rows, sh, lut, lut_n, shift, dst, smem);
    }
}

}  // namespace

// FastNlMeansDenoisingInvoker's constructor: the fixed-point weight table for 3 channels of 8 bits.
// mult = INT_MAX / (sw^2 * 255); shift = least p with 2^p >= tw^2; entry a is cvRound(mult * exp(-a * 2^shift / tw^2 / den)) with
// den = float(h * h) * 3 in float arithmetic, 1 where that is NaN (h = 0, a = 0), and 0 below 0.001 * mult.
std::vector<int> denoise_weights(float h, int tw, int sw, int* shift_out) {
    const int mult = std::min(INT_MAX / (sw * sw * 255), INT_MAX);
    int shift = 0;
    while ((1 << shift) < tw * tw) ++shift;
    const double m = (double)(1 << shift) / (tw * tw);
    const int amax = (int)(255 * 255 * 3 / m + 1);
    const float hh = h * h, den = hh * 3.0f;
    std::vector<int> lut(amax);
    for (int a = 0; a < amax; ++a) {
        const double d = a * m;
        double w = std::exp(-d / den);
        if (std::isnan(w)) w = 1.0;
        int v = (int)std::nearbyint(mult * w);         // cvRound: round half to even in the default rounding mode
        if (v < 0.001 * mult) v = 0;
        lut[a] = v;
    }
    *shift_out = shift;
    return lut;
}

}  // namespace poppy

extern "C" {

int poppy_cuda_denoise(int device, const uint8_t* src, size_t src_step, int cols, int rows, float h, int template_window_size,
                       int search_window_size, uint8_t* dst, size_t dst_step) {
    using namespace poppy;
    auto fail = [](int code, const std::string& msg) { margin_set_error("denoise: " + msg); return code; };
    if (!src || !dst || cols < 1 || rows < 1 || src_step < (size_t)cols * 3 || dst_step < (size_t)cols * 3)
        return fail(POPPY_CUDA_ERR_INVALID, "bad argument");
    if (template_window_size < 1 || search_window_size < 1 || !std::isfinite(h))
        return fail(POPPY_CUDA_ERR_INVALID, "window sizes must be >= 1 and h finite");
    const int th = template_window_size / 2, sh = search_window_size / 2;
    if (th > NL_MAX_TH || sh > NL_MAX_SH)
        return fail(POPPY_CUDA_ERR_INVALID, "template_window_size <= 15 and search_window_size <= 63 (after rounding up to odd)");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev < 1 || device < 0 || device >= n_dev)
        return fail(POPPY_CUDA_ERR_NO_DEVICE, "no such CUDA device (there is no CPU fallback)");

    int shift = 0;
    std::vector<int> lut = denoise_weights(h, 2 * th + 1, 2 * sh + 1, &shift);
    const int lut_n = (int)(std::find(lut.begin(), lut.end(), 0) - lut.begin());
    lut.resize(lut_n + 1, 0);                            // the non-zero prefix and one 0, the target of the clamp

    uint8_t *d_src = nullptr, *d_dst = nullptr;
    int* d_lut = nullptr;
#define NL_TRY(expr)                                                                                                  \
    do {                                                                                                              \
        cudaError_t e_ = (expr);                                                                                      \
        if (e_ != cudaSuccess) {                                                                                      \
            cudaFree(d_src); cudaFree(d_dst); cudaFree(d_lut);                                                        \
            return fail(POPPY_CUDA_ERR_CUDA, cudaGetErrorString(e_));                                                 \
        }                                                                                                             \
    } while (0)
    NL_TRY(cudaSetDevice(device));
    int smem_optin = 0;
    NL_TRY(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    const size_t smem_base = denoise_smem_bytes(th, sh, 0), smem_lut = denoise_smem_bytes(th, sh, lut.size());
    const bool lut_in_smem = smem_lut <= (size_t)smem_optin;     // else the table is read through L1
    const size_t pitch = (size_t)cols * 3;
    NL_TRY(cudaMalloc((void**)&d_src, pitch * rows));
    NL_TRY(cudaMalloc((void**)&d_dst, pitch * rows));
    NL_TRY(cudaMalloc((void**)&d_lut, lut.size() * sizeof(int)));
    NL_TRY(cudaMemcpy(d_lut, lut.data(), lut.size() * sizeof(int), cudaMemcpyHostToDevice));
    NL_TRY(cudaMemcpy2D(d_src, pitch, src, src_step, pitch, rows, cudaMemcpyHostToDevice));
    NL_TRY(lut_in_smem ? launch_denoise<true>(th, d_src, cols, rows, sh, d_lut, lut_n, shift, d_dst, smem_lut)
                       : launch_denoise<false>(th, d_src, cols, rows, sh, d_lut, lut_n, shift, d_dst, smem_base));
    NL_TRY(cudaMemcpy2D(dst, dst_step, d_dst, pitch, pitch, rows, cudaMemcpyDeviceToHost));
#undef NL_TRY
    cudaFree(d_src); cudaFree(d_dst); cudaFree(d_lut);
    return 0;
}

}  // extern "C"
