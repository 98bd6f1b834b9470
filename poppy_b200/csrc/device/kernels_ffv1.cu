// Output side: rendered BGR ring slots -> FFV1 packets (version 3, range coder, RGB via RCT; poppy_b200/csrc/ffv1_format.hpp,
// DESIGN §9.1). Three steps per piece of frames, all on the copy stream:
//   k_ffv1_symbols  one thread per pixel: RCT, median prediction and the quantised context of its three samples, written as
//                   (context << 16 | 16-bit folded residual) in each slice's coding order (rows, per row G', B', R').
//                   Prediction reads source samples, so every sample is independent.
//   k_ffv1_code     one thread per slice: the adaptive range coder, serial over the slice, its 2 x 666 x 32 state bytes and
//                   the transition tables in shared memory. Writes into a fixed-capacity slot; a slice that would not fit
//                   stops, is listed, and is coded again by the same kernel into worst-case scratch (ffv1::kWorst...).
//   k_ffv1_scan /   slice offsets and packet sizes (one block), then each slice's bytes and its 24-bit size copied into
//   k_ffv1_pack     contiguous per-frame packets.
#include "kernels.cuh"
#include "../ffv1_format.hpp"

namespace poppy {
namespace {

constexpr int SYM_THREADS = 128;
constexpr int SCAN_THREADS = 1024;
constexpr int PACK_THREADS = 256;
constexpr int SYM_AHEAD = 8;        // symbols the coder loads ahead of the one it codes

struct SliceRect { int x0, y0, sw, sh; };

__device__ __forceinline__ SliceRect slice_rect(int s, int w, int h, int nh, int nv) {
    const int i = s % nh, j = s / nh;
    const int x0 = (int)((int64_t)w * i / nh), y0 = (int)((int64_t)h * j / nv);
    return {x0, y0, (int)((int64_t)w * (i + 1) / nh) - x0, (int)((int64_t)h * (j + 1) / nv) - y0};
}

// JPEG2000-RCT of one BGR pixel: G' = G + ((B - G + R - G) >> 2), B' = B - G + 256, R' = R - G + 256
__device__ __forceinline__ void rct(const uint8_t* p, int out[3]) {
    const int b = p[0], g = p[1], r = p[2];
    out[0] = g + ((b - g + r - g) >> 2);
    out[1] = b - g + 256;
    out[2] = r - g + 256;
}

__device__ __forceinline__ int median3(int a, int b, int c) { return max(min(a, b), min(max(a, b), c)); }

}  // namespace

// grid (ceil(w / SYM_THREADS), h, frames)
__global__ void __launch_bounds__(SYM_THREADS) k_ffv1_symbols(const uint8_t* __restrict__ ring, size_t frame_bytes, int first_slot,
                                                              uint32_t* __restrict__ sym, int w, int h, int nh, int nv) {
    const int x = blockIdx.x * SYM_THREADS + threadIdx.x;
    if (x >= w) return;
    const int y = blockIdx.y;
    const uint8_t* frame = ring + (size_t)(first_slot + (int)blockIdx.z) * frame_bytes;
    const size_t row = (size_t)w * 3;
    // the slice holding (x, y): column i with w * i / nh <= x < w * (i + 1) / nh, likewise the row
    const int i = (int)(((int64_t)(x + 1) * nh - 1) / w), j = (int)(((int64_t)(y + 1) * nv - 1) / h);
    const SliceRect r = slice_rect(j * nh + i, w, h, nh, nv);
    const int lx = x - r.x0, ly = y - r.y0;
    int P[3], L[3], T[3] = {0, 0, 0}, LT[3] = {0, 0, 0}, RT[3] = {0, 0, 0};
    rct(frame + y * row + (size_t)x * 3, P);
    // above the slice's first row every neighbour is 0; left of its first column L is the sample above and LT the one two
    // rows up; right of its last column RT repeats the sample above (libavcodec's two-line sample ring)
    if (ly > 0) {
        rct(frame + (y - 1) * row + (size_t)x * 3, T);
        if (lx + 1 < r.sw) rct(frame + (y - 1) * row + (size_t)(x + 1) * 3, RT);
        else for (int k = 0; k < 3; ++k) RT[k] = T[k];
        if (lx > 0) rct(frame + (y - 1) * row + (size_t)(x - 1) * 3, LT);
        else if (ly > 1) rct(frame + (y - 2) * row + (size_t)x * 3, LT);
    }
    if (lx > 0) rct(frame + y * row + (size_t)(x - 1) * 3, L);
    else for (int k = 0; k < 3; ++k) L[k] = T[k];
    uint32_t* out = sym + (size_t)blockIdx.z * ((size_t)w * h * 3) + ((size_t)r.y0 * w + (size_t)r.x0 * r.sh) * 3 +
                    (size_t)ly * 3 * r.sw + lx;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        int ctx = ffv1::quant11(L[k] - LT[k]) + 11 * ffv1::quant11(LT[k] - T[k]) + 121 * ffv1::quant11(T[k] - RT[k]);
        int d = P[k] - median3(L[k], L[k] + T[k] - LT[k], T[k]);
        if (ctx < 0) { ctx = -ctx; d = -d; }
        d = ((d + 256) & 511) - 256;
        out[(size_t)k * r.sw] = ((uint32_t)ctx << 16) | (uint16_t)(int16_t)d;
    }
}

namespace {

// libavcodec's range encoder (rangecoder.h): 16-bit range, carry resolved through one outstanding byte and a run of 0xFF.
struct RangeCoder {
    uint32_t low, range;
    int outstanding_byte;
    uint32_t outstanding_count;
    uint8_t* out;
    uint32_t pos;
    const uint8_t* zero;
    const uint8_t* one;

    __device__ __forceinline__ void renorm() {
        while (range < 0x100) {
            if (outstanding_byte < 0) {
                outstanding_byte = (int)(low >> 8);
            } else if (low <= 0xFF00) {
                out[pos++] = (uint8_t)outstanding_byte;
                for (; outstanding_count; --outstanding_count) out[pos++] = 0xFF;
                outstanding_byte = (int)(low >> 8);
            } else if (low >= 0x10000) {
                out[pos++] = (uint8_t)(outstanding_byte + 1);
                for (; outstanding_count; --outstanding_count) out[pos++] = 0x00;
                outstanding_byte = (int)(low >> 8) - 0x100;
            } else {
                ++outstanding_count;
            }
            low = (low & 0xFF) << 8;
            range <<= 8;
        }
    }
    __device__ __forceinline__ void bit(uint8_t* st, int b) {
        const uint32_t s = *st;
        const uint32_t r1 = (range * s) >> 8;
        if (!b) { range -= r1; *st = zero[s]; }
        else { low += range - r1; range = r1; *st = one[s]; }
        if (range < 0x100) renorm();
    }
    // put_symbol for |v| < 512: zero flag, exponent in unary, mantissa below the leading 1, sign
    __device__ __forceinline__ void symbol(uint8_t* st, int v, bool is_signed) {
        if (v == 0) { bit(st, 1); return; }
        const int a = v < 0 ? -v : v;
        const int e = 31 - __clz(a);
        bit(st, 0);
        for (int i = 0; i < e; ++i) bit(st + 1 + i, 1);
        bit(st + 1 + e, 0);
        for (int i = e - 1; i >= 0; --i) bit(st + 22 + i, (a >> i) & 1);
        if (is_signed) bit(st + 11 + e, v < 0);
    }
    // ff_rac_terminate(c, 1)
    __device__ __forceinline__ void terminate() {
        uint8_t s = 129;
        bit(&s, 0);
        range = 0xFF; low += 0xFF; renorm();
        range = 0xFF; renorm();
    }
    // bytes out + the outstanding ones: every renormalisation step accounts for exactly one byte
    __device__ __forceinline__ uint32_t committed() const { return pos + outstanding_count + (outstanding_byte >= 0 ? 1 : 0); }
};

}  // namespace

// One thread per slice, one slice per block (the states fill 42.6 KB of shared memory). Slice t of the piece is slice
// t % slices of frame t / slices; `list` (when not null) names the slices to code instead. Its bytes go to
// out + t * cap (cap bytes), or out + k * cap for list entry k. sizes[t] = byte count, or ~0u if the slice would not fit:
// then it is appended to overflow_list. slot_of[t] = -1, or k when it was coded as list entry k.
__global__ void __launch_bounds__(1) k_ffv1_code(const uint32_t* __restrict__ sym, const uint8_t* __restrict__ tables,
                                                 int w, int h, int nh, int nv, const int* __restrict__ list, uint8_t* out,
                                                 size_t cap, uint32_t* sizes, int* slot_of, int* overflow_count,
                                                 int* overflow_list) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint8_t* zero = smem;
    uint8_t* one = smem + 256;
    uint8_t* states = smem + 512;
    const int t = list ? list[blockIdx.x] : (int)blockIdx.x;
    const int slices = nh * nv, f = t / slices, s = t % slices;
    const SliceRect r = slice_rect(s, w, h, nh, nv);
    slot_of[t] = list ? (int)blockIdx.x : -1;
    for (int i = 0; i < 32; ++i) reinterpret_cast<uint4*>(smem)[i] = reinterpret_cast<const uint4*>(tables)[i];
    const uint4 init = make_uint4(0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u);
    for (int i = 0; i < 2 * ffv1::kContexts * ffv1::kStateBytes / 16; ++i) reinterpret_cast<uint4*>(states)[i] = init;

    RangeCoder rc{0, 0xFF00, -1, 0, out + (size_t)blockIdx.x * cap, 0, zero, one};
    uint8_t* hdr = states + 2 * ffv1::kContexts * ffv1::kStateBytes;       // the slice header's own 32 states
    for (int i = 0; i < 32; ++i) hdr[i] = 128;
    if (s == 0) { uint8_t key = 128; rc.bit(&key, 1); }       // keyframe
    rc.symbol(hdr, s % nh, false);                            // slice_x, slice_y
    rc.symbol(hdr, s / nh, false);
    rc.symbol(hdr, 0, false);                                 // slice width and height - 1, in slice units
    rc.symbol(hdr, 0, false);
    rc.symbol(hdr, 0, false);                                 // quant-table set of both context planes
    rc.symbol(hdr, 0, false);
    rc.symbol(hdr, 3, false);                                 // picture_structure: progressive
    rc.symbol(hdr, 0, false);                                 // sample aspect ratio 0:0
    rc.symbol(hdr, 0, false);

    const uint32_t* p = sym + (size_t)f * ((size_t)w * h * 3) + ((size_t)r.y0 * w + (size_t)r.x0 * r.sh) * 3;
    // a symbol takes at most 19 renormalisation steps (one per decision: every state lies in [8, 248], so a decision keeps
    // at least 8 / 256 of the range), the termination 3
    const size_t limit = cap >= 22 + 3 ? cap - 22 - 3 : 0;
    // symbols in coding order (per row G', B', R'), read 8 ahead: the loads of the next group are in flight while the
    // serial coder works through the current one
    const size_t n = (size_t)r.sw * r.sh * 3;
    uint32_t cur[SYM_AHEAD];
#pragma unroll
    for (int j = 0; j < SYM_AHEAD; ++j) cur[j] = (size_t)j < n ? __ldg(p + j) : 0u;
    int x = 0, plane = 0;
    for (size_t base = 0; base < n; base += SYM_AHEAD) {
        uint32_t next[SYM_AHEAD];
#pragma unroll
        for (int j = 0; j < SYM_AHEAD; ++j) next[j] = base + SYM_AHEAD + j < n ? __ldg(p + base + SYM_AHEAD + j) : 0u;
#pragma unroll
        for (int j = 0; j < SYM_AHEAD; ++j) {
            if (base + j >= n) break;
            if (rc.committed() > limit) {
                sizes[t] = ~0u;
                overflow_list[atomicAdd(overflow_count, 1)] = t;
                return;
            }
            uint8_t* st = states + (plane ? ffv1::kContexts * ffv1::kStateBytes : 0);
            rc.symbol(st + (cur[j] >> 16) * ffv1::kStateBytes, (int16_t)(cur[j] & 0xFFFF), true);
            if (++x == r.sw) { x = 0; plane = plane == 2 ? 0 : plane + 1; }
        }
#pragma unroll
        for (int j = 0; j < SYM_AHEAD; ++j) cur[j] = next[j];
    }
    rc.terminate();
    sizes[t] = rc.pos;
}

// One block: packet offsets of the piece's slices (each slice's bytes + its 3-byte size), and the packet size per frame.
__global__ void __launch_bounds__(SCAN_THREADS) k_ffv1_scan(const uint32_t* __restrict__ sizes, int slices, int frames,
                                                            uint64_t* __restrict__ offsets, uint32_t* __restrict__ frame_sizes) {
    __shared__ uint64_t part[SCAN_THREADS];
    const int n = slices * frames;
    const int per = (n + SCAN_THREADS - 1) / SCAN_THREADS;
    const int lo = min(n, (int)threadIdx.x * per), hi = min(n, lo + per);
    uint64_t sum = 0;
    for (int i = lo; i < hi; ++i) sum += sizes[i] + 3;
    part[threadIdx.x] = sum;
    __syncthreads();
    for (int d = 1; d < SCAN_THREADS; d <<= 1) {
        const uint64_t v = threadIdx.x >= (unsigned)d ? part[threadIdx.x - d] : 0;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    uint64_t off = part[threadIdx.x] - sum;
    for (int i = lo; i < hi; ++i) { offsets[i] = off; off += sizes[i] + 3; }
    if (threadIdx.x == SCAN_THREADS - 1) offsets[n] = part[threadIdx.x];
    __syncthreads();
    for (int f = threadIdx.x; f < frames; f += SCAN_THREADS)
        frame_sizes[f] = (uint32_t)(offsets[(size_t)(f + 1) * slices] - offsets[(size_t)f * slices]);
}

// grid (slices of the piece): slice t's bytes from its slot (or from the overflow scratch) + its 24-bit size, big-endian.
__global__ void __launch_bounds__(PACK_THREADS) k_ffv1_pack(const uint8_t* __restrict__ slots, size_t cap,
                                                            const uint8_t* __restrict__ scratch, size_t scratch_cap,
                                                            const int* __restrict__ slot_of, const uint32_t* __restrict__ sizes,
                                                            const uint64_t* __restrict__ offsets, uint8_t* __restrict__ packets) {
    const int t = blockIdx.x;
    const uint32_t n = sizes[t];
    const int k = slot_of[t];
    const uint8_t* src = k < 0 ? slots + (size_t)t * cap : scratch + (size_t)k * scratch_cap;
    uint8_t* dst = packets + offsets[t];
    for (uint32_t i = threadIdx.x; i < n; i += PACK_THREADS) dst[i] = src[i];
    if (threadIdx.x < 3) dst[n + threadIdx.x] = (uint8_t)(n >> (16 - 8 * threadIdx.x));
}

size_t ffv1_code_smem() { return 512 + 2 * ffv1::kContexts * ffv1::kStateBytes + 32; }

void launch_ffv1_symbols(cudaStream_t st, const uint8_t* ring, size_t frame_bytes, int first_slot, int frames, uint32_t* sym, int w,
                         int h, int nh, int nv) {
    const dim3 grid((unsigned)div_up(w, SYM_THREADS), (unsigned)h, (unsigned)frames);
    k_ffv1_symbols<<<grid, SYM_THREADS, 0, st>>>(ring, frame_bytes, first_slot, sym, w, h, nh, nv);
}

cudaError_t launch_ffv1_code(cudaStream_t st, const uint32_t* sym, const uint8_t* tables, int w, int h, int nh, int nv, int count,
                             const int* list, uint8_t* out, size_t cap, uint32_t* sizes, int* slot_of, int* overflow_count,
                             int* overflow_list) {
    static_assert(2 * ffv1::kContexts * ffv1::kStateBytes % 16 == 0, "states are set in 16-byte words");
    const size_t smem = ffv1_code_smem();
    if (cudaError_t e = cudaFuncSetAttribute(k_ffv1_code, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) return e;
    k_ffv1_code<<<(unsigned)count, 1, smem, st>>>(sym, tables, w, h, nh, nv, list, out, cap, sizes, slot_of, overflow_count,
                                                        overflow_list);
    return cudaGetLastError();
}

void launch_ffv1_pack(cudaStream_t st, const uint32_t* sizes, int slices, int frames, uint64_t* offsets, uint32_t* frame_sizes,
                      const uint8_t* slots, size_t cap, const uint8_t* scratch, size_t scratch_cap, const int* slot_of,
                      uint8_t* packets) {
    k_ffv1_scan<<<1, SCAN_THREADS, 0, st>>>(sizes, slices, frames, offsets, frame_sizes);
    k_ffv1_pack<<<(unsigned)(slices * frames), PACK_THREADS, 0, st>>>(slots, cap, scratch, scratch_cap, slot_of, sizes, offsets,
                                                                     packets);
}

}  // namespace poppy
