// A minimal Matroska writer for FFV1 packets (include/poppy_host.h, poppy_host_mkv_*): the layout libavformat writes for
// cv2.VideoWriter("x.mkv", FFV1): EBML header, one Segment with Info and one video track (CodecID "V_FFV1", CodecPrivate =
// the configuration record), then Clusters of SimpleBlocks, every block a keyframe. Timestamps are in milliseconds; a new
// Cluster starts before a block's 16-bit relative timestamp would overflow. Sizes of the Segment and of each Cluster are
// written as 8-byte placeholders and patched, with the Duration, when they are known. No Cues: players read it
// sequentially, as the reference's output is read.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../../include/poppy_host.h"

struct poppy_host_mkv {
    FILE* f = nullptr;
    long long segment_data = 0, duration_pos = 0, cluster_size_pos = -1;
    long long cluster_ts = 0;
    long long frames = 0;
    double frame_ms = 0;
    bool failed = false;
};

namespace {

void put(std::vector<uint8_t>& b, uint64_t v, int n) { for (int k = n - 1; k >= 0; --k) b.push_back((uint8_t)(v >> (8 * k))); }
void put_id(std::vector<uint8_t>& b, uint32_t id) { put(b, id, id > 0xFFFFFF ? 4 : id > 0xFFFF ? 3 : id > 0xFF ? 2 : 1); }
void put_size8(std::vector<uint8_t>& b, uint64_t n) { put(b, (1ULL << 56) | n, 8); }  // 8-byte size vint
void put_size(std::vector<uint8_t>& b, uint64_t n) {
    if (n < 0x7F) put(b, 0x80 | n, 1);
    else if (n < 0x3FFF) put(b, 0x4000 | n, 2);
    else if (n < 0x1FFFFF) put(b, 0x200000 | n, 3);
    else if (n < 0x0FFFFFFF) put(b, 0x10000000 | n, 4);
    else put_size8(b, n);
}
void element(std::vector<uint8_t>& b, uint32_t id, const std::vector<uint8_t>& payload) {
    put_id(b, id); put_size(b, payload.size()); b.insert(b.end(), payload.begin(), payload.end());
}
void uint_el(std::vector<uint8_t>& b, uint32_t id, uint64_t v) {
    int n = 1;
    while (n < 8 && (v >> (8 * n))) ++n;
    std::vector<uint8_t> p;
    put(p, v, n);
    element(b, id, p);
}
void str_el(std::vector<uint8_t>& b, uint32_t id, const std::string& s) { element(b, id, std::vector<uint8_t>(s.begin(), s.end())); }
std::vector<uint8_t> f64(double v) {
    uint64_t u;
    std::memcpy(&u, &v, 8);
    std::vector<uint8_t> p;
    put(p, u, 8);
    return p;
}

bool write_all(poppy_host_mkv* m, const std::vector<uint8_t>& b) {
    if (!m->failed && std::fwrite(b.data(), 1, b.size(), m->f) != b.size()) m->failed = true;
    return !m->failed;
}
bool patch(poppy_host_mkv* m, long long pos, const std::vector<uint8_t>& b) {
    const long long here = std::ftell(m->f);
    if (std::fseek(m->f, pos, SEEK_SET) != 0) return !(m->failed = true);
    write_all(m, b);
    if (std::fseek(m->f, here, SEEK_SET) != 0) m->failed = true;
    return !m->failed;
}
bool close_cluster(poppy_host_mkv* m) {
    if (m->cluster_size_pos < 0) return true;
    std::vector<uint8_t> s;
    put_size8(s, (uint64_t)(std::ftell(m->f) - m->cluster_size_pos - 8));
    const long long pos = m->cluster_size_pos;
    m->cluster_size_pos = -1;
    return patch(m, pos, s);
}

}  // namespace

extern "C" {

int poppy_host_mkv_open(poppy_host_mkv** out, const char* path, int width, int height, int fps_num, int fps_den) {
    if (!out) return POPPY_CUDA_ERR_INVALID;
    *out = nullptr;
    if (!path || width < 1 || height < 1 || fps_num < 1 || fps_den < 1) return POPPY_CUDA_ERR_INVALID;
    std::vector<uint8_t> rec(256);
    size_t rec_size = 0;
    if (int rc = poppy_host_ffv1_config(width, height, rec.data(), rec.size(), &rec_size)) return rc;
    rec.resize(rec_size);
    FILE* f = std::fopen(path, "wb");
    if (!f) return POPPY_CUDA_ERR_INVALID;
    auto* m = new poppy_host_mkv();
    m->f = f;
    m->frame_ms = 1000.0 * fps_den / fps_num;

    std::vector<uint8_t> b, hdr;
    uint_el(hdr, 0x4286, 1);                   // EBMLVersion
    uint_el(hdr, 0x42F7, 1);                   // EBMLReadVersion
    uint_el(hdr, 0x42F2, 4);                   // EBMLMaxIDLength
    uint_el(hdr, 0x42F3, 8);                   // EBMLMaxSizeLength
    str_el(hdr, 0x4282, "matroska");           // DocType
    uint_el(hdr, 0x4287, 4);                   // DocTypeVersion
    uint_el(hdr, 0x4285, 2);                   // DocTypeReadVersion
    element(b, 0x1A45DFA3, hdr);
    put_id(b, 0x18538067);                     // Segment, size patched on close
    put_size8(b, 0);
    m->segment_data = (long long)b.size();

    std::vector<uint8_t> info;
    uint_el(info, 0x2AD7B1, 1000000);          // TimestampScale: 1 ms
    str_el(info, 0x4D80, "poppy_b200");        // MuxingApp
    str_el(info, 0x5741, "poppy_b200");        // WritingApp
    put_id(info, 0x4489);                      // Duration (float64, ms), patched on close
    put_size(info, 8);
    const size_t duration_in_info = info.size();
    const std::vector<uint8_t> zero = f64(0.0);
    info.insert(info.end(), zero.begin(), zero.end());
    put_id(b, 0x1549A966);
    put_size(b, info.size());
    m->duration_pos = (long long)(b.size() + duration_in_info);
    b.insert(b.end(), info.begin(), info.end());

    std::vector<uint8_t> video, track, tracks;
    uint_el(video, 0xB0, (uint64_t)width);     // PixelWidth
    uint_el(video, 0xBA, (uint64_t)height);    // PixelHeight
    uint_el(track, 0xD7, 1);                   // TrackNumber
    uint_el(track, 0x73C5, 1);                 // TrackUID
    uint_el(track, 0x9C, 0);                   // FlagLacing
    str_el(track, 0x86, "V_FFV1");             // CodecID
    uint_el(track, 0x83, 1);                   // TrackType: video
    uint_el(track, 0x23E383, (uint64_t)std::llround(1e9 * fps_den / fps_num));   // DefaultDuration (ns)
    element(track, 0xE0, video);
    element(track, 0x63A2, rec);               // CodecPrivate: the FFV1 configuration record
    element(tracks, 0xAE, track);
    element(b, 0x1654AE6B, tracks);
    if (!write_all(m, b)) { std::fclose(f); delete m; return POPPY_CUDA_ERR_INVALID; }
    *out = m;
    return 0;
}

int poppy_host_mkv_write(poppy_host_mkv* m, const uint8_t* packet, size_t size) {
    if (!m || !packet || size == 0 || m->failed) return POPPY_CUDA_ERR_INVALID;
    const long long ts = std::llround(m->frames * m->frame_ms);
    std::vector<uint8_t> b;
    if (m->cluster_size_pos < 0 || ts - m->cluster_ts > 32767) {
        if (!close_cluster(m)) return POPPY_CUDA_ERR_INVALID;
        put_id(b, 0x1F43B675);                 // Cluster, size patched when the next one starts or on close
        put_size8(b, 0);
        m->cluster_size_pos = std::ftell(m->f) + 4;
        m->cluster_ts = ts;
        uint_el(b, 0xE7, (uint64_t)ts);        // Cluster Timestamp
    }
    put_id(b, 0xA3);                           // SimpleBlock: track 1, relative timestamp, keyframe flag
    put_size(b, size + 4);
    put(b, 0x81, 1);
    put(b, (uint16_t)(int16_t)(ts - m->cluster_ts), 2);
    put(b, 0x80, 1);
    b.insert(b.end(), packet, packet + size);
    if (!write_all(m, b)) return POPPY_CUDA_ERR_INVALID;
    ++m->frames;
    return 0;
}

int poppy_host_mkv_close(poppy_host_mkv* m) {
    if (!m) return POPPY_CUDA_ERR_INVALID;
    bool ok = close_cluster(m);
    const long long end = std::ftell(m->f);
    std::vector<uint8_t> s;
    put_size8(s, (uint64_t)(end - m->segment_data));
    ok = ok && patch(m, m->segment_data - 8, s) && patch(m, m->duration_pos, f64(m->frames * m->frame_ms));
    ok = std::fclose(m->f) == 0 && ok && !m->failed;
    delete m;
    return ok ? 0 : POPPY_CUDA_ERR_INVALID;
}

}  // extern "C"
