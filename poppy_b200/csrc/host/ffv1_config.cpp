// FFV1 configuration record (the codec's extradata, Matroska CodecPrivate) of the streams poppy_cuda_download_ffv1 writes:
// the fields of ffv1_format.hpp, range coded with the default state table and one context of 32 states, terminated as
// libavcodec terminates it and followed by its CRC-32 (MSB first, polynomial 0x04C11DB7, init 0), big-endian.
#include <cstring>
#include <vector>

#include "../../../include/poppy_host.h"
#include "../ffv1_format.hpp"

namespace {

struct HostRangeCoder {
    std::vector<uint8_t> out;
    uint32_t low = 0, range = 0xFF00, outstanding_count = 0;
    int outstanding_byte = -1;
    uint8_t zero[256], one[256];
    HostRangeCoder() { poppy::ffv1::build_states(zero, one); }

    void renorm() {
        while (range < 0x100) {
            if (outstanding_byte < 0) {
                outstanding_byte = (int)(low >> 8);
            } else if (low <= 0xFF00) {
                out.push_back((uint8_t)outstanding_byte);
                for (; outstanding_count; --outstanding_count) out.push_back(0xFF);
                outstanding_byte = (int)(low >> 8);
            } else if (low >= 0x10000) {
                out.push_back((uint8_t)(outstanding_byte + 1));
                for (; outstanding_count; --outstanding_count) out.push_back(0x00);
                outstanding_byte = (int)(low >> 8) - 0x100;
            } else {
                ++outstanding_count;
            }
            low = (low & 0xFF) << 8;
            range <<= 8;
        }
    }
    void bit(uint8_t* st, int b) {
        const uint32_t r1 = (range * *st) >> 8;
        if (!b) { range -= r1; *st = zero[*st]; }
        else { low += range - r1; range = r1; *st = one[*st]; }
        renorm();
    }
    void symbol(uint8_t* st, int v) {          // unsigned
        if (v == 0) { bit(st, 1); return; }
        int e = 0;
        while ((v >> (e + 1)) != 0) ++e;
        bit(st, 0);
        for (int i = 0; i < e; ++i) bit(st + 1 + (i < 9 ? i : 9), 1);
        bit(st + 1 + (e < 9 ? e : 9), 0);
        for (int i = e - 1; i >= 0; --i) bit(st + 22 + (i < 9 ? i : 9), (v >> i) & 1);
    }
    void terminate() {
        uint8_t s = 129;
        bit(&s, 0);
        range = 0xFF; low += 0xFF; renorm();
        range = 0xFF; renorm();
    }
};

// run lengths of a quant table's non-negative half (indices 0..127), as libavcodec's write_quant_table codes them
void write_quant_table(HostRangeCoder& rc, int scale) {
    uint8_t st[32];
    std::memset(st, 128, sizeof st);
    int last = 0;
    for (int i = 1; i < 128; ++i)
        if (scale * poppy::ffv1::quant11(i) != scale * poppy::ffv1::quant11(i - 1)) { rc.symbol(st, i - last - 1); last = i; }
    rc.symbol(st, 128 - last - 1);
}

uint32_t crc32_msb(const uint8_t* p, size_t n) {
    uint32_t crc = 0;
    for (size_t i = 0; i < n; ++i) {
        crc ^= (uint32_t)p[i] << 24;
        for (int k = 0; k < 8; ++k) crc = (crc & 0x80000000u) ? (crc << 1) ^ 0x04C11DB7u : crc << 1;
    }
    return crc;
}

}  // namespace

extern "C" int poppy_host_ffv1_config(int width, int height, uint8_t* dst, size_t cap, size_t* size) {
    if (width < 1 || height < 1 || !size) return POPPY_CUDA_ERR_INVALID;
    int nh = 0, nv = 0;
    poppy::ffv1::slice_grid(width, height, &nh, &nv);
    HostRangeCoder rc;
    uint8_t st[32];
    std::memset(st, 128, sizeof st);
    for (int v : {3, 4, 1, 1, 8}) rc.symbol(st, v);    // version, micro_version, coder_type, colorspace_type, bits
    rc.bit(st, 1);                                     // chroma_planes
    rc.symbol(st, 0);                                  // no chroma subsampling
    rc.symbol(st, 0);
    rc.bit(st, 0);                                     // no alpha plane
    rc.symbol(st, nh - 1);
    rc.symbol(st, nv - 1);
    rc.symbol(st, 1);                                  // one quant-table set: quant11, 11 * quant11, 121 * quant11, 0, 0
    for (int scale : {1, 11, 121, 0, 0}) write_quant_table(rc, scale);
    rc.bit(st, 0);                                     // initial states not coded: all 128
    rc.symbol(st, 0);                                  // ec: no slice CRCs
    rc.symbol(st, 1);                                  // intra
    rc.terminate();
    const uint32_t crc = crc32_msb(rc.out.data(), rc.out.size());
    for (int k = 3; k >= 0; --k) rc.out.push_back((uint8_t)(crc >> (8 * k)));
    *size = rc.out.size();
    if (!dst || cap < rc.out.size()) return POPPY_CUDA_ERR_INVALID;
    std::memcpy(dst, rc.out.data(), rc.out.size());
    return 0;
}
