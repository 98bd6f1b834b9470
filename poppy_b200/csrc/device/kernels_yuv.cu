// Output side: rendered BGR ring slots -> packed I420 (YUV 4:2:0) frames, byte for byte what
// cv::cvtColor(bgr, out, COLOR_BGR2YUV_I420) gives (OpenCV 4.13, imgproc/src/color_yuv.simd.hpp, RGB888toYUV420pInvoker):
//   Y = sat_u8((269484 R + 528482 G + 102760 B + 2^19 + (16 << 20)) >> 20)                     every pixel
//   U = sat_u8((-155188 R - 305135 G + 460324 B + 2^19 + (128 << 20)) >> 20)                   pixel (2i, 2j) only
//   V = sat_u8(( 460324 R - 385875 G -  74448 B + 2^19 + (128 << 20)) >> 20)                   pixel (2i, 2j) only
// in int32 with an arithmetic shift. Chroma is the top-left pixel of each 2 x 2 block, not an average. Layout of one frame:
// the Y plane (W x H), then U and V ((W/2) x (H/2) each), all rows tightly packed: W * H * 3 / 2 bytes.
#include "kernels.cuh"

namespace poppy {
namespace {

constexpr int I420_THREADS = 128;

__device__ __forceinline__ uint32_t sat_u8(int v) { return (uint32_t)min(max(v, 0), 255); }
__device__ __forceinline__ uint32_t luma(int b, int g, int r) {
    return sat_u8((269484 * r + 528482 * g + 102760 * b + (1 << 19) + (16 << 20)) >> 20);
}
__device__ __forceinline__ uint32_t chroma_u(int b, int g, int r) {
    return sat_u8((-155188 * r - 305135 * g + 460324 * b + (1 << 19) + (128 << 20)) >> 20);
}
__device__ __forceinline__ uint32_t chroma_v(int b, int g, int r) {
    return sat_u8((460324 * r - 385875 * g - 74448 * b + (1 << 19) + (128 << 20)) >> 20);
}

template <int PX> struct I420Words;
template <> struct I420Words<2> { using Pix = uint16_t; using Chroma = uint8_t; };    // any even width
template <> struct I420Words<4> { using Pix = uint32_t; using Chroma = uint16_t; };   // width % 4 == 0: 32-bit rows

}  // namespace

// One thread: PX pixels of rows 2i and 2i+1 (3 loads of PX bytes each per row), PX luma bytes per row, PX/2 bytes of U and
// of V. Consecutive threads take consecutive pixels, so every warp reads and writes contiguous spans.
// grid (ceil(w / PX / I420_THREADS), h / 2, frames); frame f reads ring slot first_slot + f, writes out + f * w * h * 3 / 2.
template <int PX>
__global__ void __launch_bounds__(I420_THREADS) k_bgr_to_i420(const uint8_t* __restrict__ ring, size_t frame_bytes, int first_slot,
                                                             uint8_t* __restrict__ out, int w, int h) {
    using Pix = typename I420Words<PX>::Pix;
    using Chroma = typename I420Words<PX>::Chroma;
    const int x0 = (blockIdx.x * I420_THREADS + threadIdx.x) * PX;
    if (x0 >= w) return;
    const int i = blockIdx.y;
    const size_t W = (size_t)w, plane = W * (size_t)h;
    const uint8_t* src = ring + (size_t)(first_slot + (int)blockIdx.z) * frame_bytes + (size_t)(2 * i) * W * 3 + (size_t)x0 * 3;
    uint8_t* frame = out + (size_t)blockIdx.z * (plane * 3 / 2);
    uint8_t* y_out = frame + (size_t)(2 * i) * W + x0;
    Chroma* u_out = reinterpret_cast<Chroma*>(frame + plane + (size_t)i * (W / 2) + x0 / 2);
    Chroma* v_out = reinterpret_cast<Chroma*>(frame + plane + plane / 4 + (size_t)i * (W / 2) + x0 / 2);
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const Pix* s = reinterpret_cast<const Pix*>(src + r * W * 3);
        const Pix words[3] = {s[0], s[1], s[2]};
        int px[3 * PX];
#pragma unroll
        for (int k = 0; k < 3 * PX; ++k) px[k] = (words[k / PX] >> (8 * (k % PX))) & 0xff;
        Pix y = 0;
#pragma unroll
        for (int p = 0; p < PX; ++p) y |= (Pix)(luma(px[3 * p], px[3 * p + 1], px[3 * p + 2]) << (8 * p));
        *reinterpret_cast<Pix*>(y_out + r * W) = y;
        if (r == 0) {
            Chroma u = 0, v = 0;
#pragma unroll
            for (int p = 0; p < PX; p += 2) {
                u |= (Chroma)(chroma_u(px[3 * p], px[3 * p + 1], px[3 * p + 2]) << (4 * p));
                v |= (Chroma)(chroma_v(px[3 * p], px[3 * p + 1], px[3 * p + 2]) << (4 * p));
            }
            *u_out = u;
            *v_out = v;
        }
    }
}

void launch_bgr_to_i420(cudaStream_t st, const uint8_t* ring, size_t frame_bytes, int first_slot, int frames, uint8_t* out, int w,
                        int h) {
    // 32-bit words need every row start 4-byte aligned: w % 4 == 0 makes the BGR rows (3w), the luma rows (w), the chroma
    // rows (w / 2, 2-byte words) and every frame and plane offset multiples of the word size
    const bool vec = (w & 3) == 0 && (reinterpret_cast<uintptr_t>(ring) & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0;
    const int px = vec ? 4 : 2;
    const dim3 grid((unsigned)div_up(w / px, I420_THREADS), (unsigned)(h / 2), (unsigned)frames);
    if (vec) k_bgr_to_i420<4><<<grid, I420_THREADS, 0, st>>>(ring, frame_bytes, first_slot, out, w, h);
    else k_bgr_to_i420<2><<<grid, I420_THREADS, 0, st>>>(ring, frame_bytes, first_slot, out, w, h);
}

}  // namespace poppy
