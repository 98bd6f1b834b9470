"""Test-only restatement of the FFV1 stream the GPU encoder writes, plain Python and numpy (no cv2):

- FFV1 version 3, micro_version 4 (RFC 9043), range coder (coder_type 1) with the default state-transition table,
  RGB via JPEG2000-RCT (colorspace_type 1), 8 bits, no alpha, ec 0, intra 1, all initial states 128 (states_coded 0),
  one quant-table set (libavcodec's 8-bit default, context model 0) for both context planes.
- The slice grid slice_grid(w, h), a function of the frame size alone.
- A decoder of the same configuration, which also reads the configuration record and the slice headers libavcodec's
  encoder writes with coder_type 0 (Golomb-Rice content, not decoded here).
- A Matroska (EBML) reader for the files poppy_host_mkv_* and libavformat write.

The bitstream details restated here were checked against what libavcodec 62 writes and decodes (the fixture under
tests/golden/output/ffv1/ and cv2.VideoCapture on this module's own streams), not against a copy of the specification.
"""
import numpy as np

# ---- range coder ---------------------------------------------------------------------------------------------------------


def build_states(factor=int(0.05 * (1 << 32)), max_p=256 - 8):
    """(zero_state, one_state): libavcodec's ff_build_rac_states(c, 0.05 * 2^32, 248), the default transition table."""
    one = 1 << 32
    zero, ones = [0] * 256, [0] * 256
    last, p = 0, one // 2
    for _ in range(128):
        p8 = (256 * p + one // 2) >> 32
        if p8 <= last:
            p8 = last + 1
        if last and last < 256 and p8 <= max_p:
            ones[last] = p8
        p += ((one - p) * factor + one // 2) >> 32
        last = p8
    for i in range(256 - max_p, max_p + 1):
        if ones[i]:
            continue
        p = (i * one + 128) >> 8
        p += ((one - p) * factor + one // 2) >> 32
        p8 = (256 * p + one // 2) >> 32
        if p8 <= i:
            p8 = i + 1
        if p8 > max_p:
            p8 = max_p
        ones[i] = p8
    for i in range(1, 255):
        zero[i] = 256 - ones[256 - i]
    return zero, ones


ZERO_STATE, ONE_STATE = build_states()


class RangeEncoder:
    def __init__(self):
        self.out = bytearray()
        self.low, self.range = 0, 0xFF00
        self.outstanding_count, self.outstanding_byte = 0, -1

    def _renorm(self):
        while self.range < 0x100:
            if self.outstanding_byte < 0:
                self.outstanding_byte = self.low >> 8
            elif self.low <= 0xFF00:
                self.out.append(self.outstanding_byte)
                self.out.extend(b"\xff" * self.outstanding_count)
                self.outstanding_count = 0
                self.outstanding_byte = self.low >> 8
            elif self.low >= 0x10000:
                self.out.append(self.outstanding_byte + 1)
                self.out.extend(b"\x00" * self.outstanding_count)
                self.outstanding_count = 0
                self.outstanding_byte = (self.low >> 8) - 0x100
            else:
                self.outstanding_count += 1
            self.low = (self.low & 0xFF) << 8
            self.range <<= 8

    def bit(self, st, i, b):
        r1 = (self.range * st[i]) >> 8
        if not b:
            self.range -= r1
            st[i] = ZERO_STATE[st[i]]
        else:
            self.low += self.range - r1
            self.range = r1
            st[i] = ONE_STATE[st[i]]
        if self.range < 0x100:
            self._renorm()

    def symbol(self, st, v, signed):
        """put_symbol: zero flag, exponent in unary, mantissa MSB first (without its leading 1), then the sign."""
        if v == 0:
            self.bit(st, 0, 1)
            return
        a = abs(v) if signed else v
        e = a.bit_length() - 1
        self.bit(st, 0, 0)
        for i in range(e):
            self.bit(st, 1 + min(i, 9), 1)
        self.bit(st, 1 + min(e, 9), 0)
        for i in range(e - 1, -1, -1):
            self.bit(st, 22 + min(i, 9), (a >> i) & 1)
        if signed:
            self.bit(st, 11 + min(e, 10), v < 0)

    def terminate(self):
        """ff_rac_terminate(c, 1): a 0 with state 129, then flush. Returns the bytes."""
        self.bit([129], 0, 0)
        self.range = 0xFF
        self.low += 0xFF
        self._renorm()
        self.range = 0xFF
        self._renorm()
        return bytes(self.out)


class RangeDecoder:
    def __init__(self, buf, end=None):
        self.b = buf
        self.end = len(buf) if end is None else end
        self.pos = 2
        self.low = (buf[0] << 8) | buf[1]
        self.range = 0xFF00
        if self.low >= 0xFF00:
            self.low, self.end = 0xFF00, 2

    def bit(self, st, i):
        r1 = (self.range * st[i]) >> 8
        self.range -= r1
        if self.low < self.range:
            st[i] = ZERO_STATE[st[i]]
            b = 0
        else:
            self.low -= self.range
            self.range = r1
            st[i] = ONE_STATE[st[i]]
            b = 1
        if self.range < 0x100:
            self.range <<= 8
            self.low <<= 8
            if self.pos < self.end:
                self.low += self.b[self.pos]
                self.pos += 1
        return b

    def symbol(self, st, signed):
        if self.bit(st, 0):
            return 0
        e = 0
        while self.bit(st, 1 + min(e, 9)):
            e += 1
            if e > 31:
                raise ValueError("symbol exponent out of range")
        a = 1
        for i in range(e - 1, -1, -1):
            a = 2 * a + self.bit(st, 22 + min(i, 9))
        return -a if signed and self.bit(st, 11 + min(e, 10)) else a


def crc32_msb(data, crc=0):
    """libavutil's av_crc(AV_CRC_32_IEEE, 0, ...) as FFV1 stores it: polynomial 0x04C11DB7, MSB first, no reflection, init
    0, no final xor; appended big-endian, so the CRC over record + CRC is 0."""
    for byte in data:
        crc ^= byte << 24
        for _ in range(8):
            crc = ((crc << 1) ^ 0x04C11DB7) & 0xFFFFFFFF if crc & 0x80000000 else (crc << 1) & 0xFFFFFFFF
    return crc


# ---- configuration -------------------------------------------------------------------------------------------------------

# libavcodec's quant11 (ffv1enc.c), the table of its 8-bit default (context model 0), as its configuration record carries it


def _quant_from_runs(runs):
    q = np.zeros(256, np.int32)
    i = 0
    for v, n in enumerate(runs):
        q[i:i + n] = v
        i += n
    assert i == 128
    q[129:] = -q[1:128][::-1]
    q[128] = -q[127]
    return q


# run lengths of values 0, 1, 2, 3, 4, 5 over indices 0..127
QUANT11_RUN_LENGTHS = (1, 1, 3, 7, 23, 93)
QUANT11 = _quant_from_runs(QUANT11_RUN_LENGTHS)
CONTEXT_COUNT = (11 * 11 * 11 + 1) // 2        # 666: contexts q0 + 11 q1 + 121 q2, folded by sign
SLICE_PX = 128 * 96                            # target pixels per slice
MAX_SLICES_H = MAX_SLICES_V = 32               # the largest grid libavcodec 62 decodes is 1024 slices


def slice_grid(w, h):
    """(num_h_slices, num_v_slices): slices of about 128 x 96 pixels, at most 32 x 32, never more than w columns or h rows."""
    return min(w, MAX_SLICES_H, max(1, (w + 64) // 128)), min(h, MAX_SLICES_V, max(1, (h + 48) // 96))


def slice_rects(w, h, grid=None):
    """Slices in raster order as (x0, y0, x1, y1): column boundaries w * i // nh, row boundaries h * j // nv."""
    nh, nv = grid or slice_grid(w, h)
    return [(w * i // nh, h * j // nv, w * (i + 1) // nh, h * (j + 1) // nv) for j in range(nv) for i in range(nh)]


def _write_quant_table(rc, q):
    st = [128] * 32
    last = 0
    for i in range(1, 128):
        if q[i] != q[i - 1]:
            rc.symbol(st, i - last - 1, False)
            last = i
    rc.symbol(st, 128 - last - 1, False)


def config_record(w, h, grid=None):
    """The configuration record (codec extradata) of this encoder's streams at w x h."""
    nh, nv = grid or slice_grid(w, h)
    rc = RangeEncoder()
    st = [128] * 32
    for v in (3, 4, 1, 1, 8):                  # version, micro_version, coder_type, colorspace_type, bits_per_raw_sample
        rc.symbol(st, v, False)
    rc.bit(st, 0, 1)                           # chroma_planes
    rc.symbol(st, 0, False)                    # log2 h chroma subsample
    rc.symbol(st, 0, False)                    # log2 v chroma subsample
    rc.bit(st, 0, 0)                           # extra_plane (alpha)
    rc.symbol(st, nh - 1, False)
    rc.symbol(st, nv - 1, False)
    rc.symbol(st, 1, False)                    # quant_table_set_count
    zero = np.zeros(256, np.int32)
    for q in (QUANT11, 11 * QUANT11, 121 * QUANT11, zero, zero):
        _write_quant_table(rc, q)
    rc.bit(st, 0, 0)                           # states_coded
    rc.symbol(st, 0, False)                    # ec
    rc.symbol(st, 1, False)                    # intra
    rec = rc.terminate()
    return rec + crc32_msb(rec).to_bytes(4, "big")


def _read_quant_table(rd, scale):
    st = [128] * 32
    q = np.zeros(256, np.int32)
    i, v = 0, 0
    while i < 128:
        n = rd.symbol(st, False) + 1
        if n > 128 - i:
            raise ValueError("bad quant table")
        q[i:i + n] = scale * v
        i += n
        v += 1
    q[129:] = -q[1:128][::-1]
    q[128] = -q[127]
    return q, 2 * v - 1


def parse_config(rec):
    """The fields of a configuration record (version 3), as libavcodec's read_extra_header reads them."""
    if crc32_msb(rec) != 0:
        raise ValueError("configuration record CRC mismatch")
    rd = RangeDecoder(rec, len(rec) - 4)
    st = [128] * 32
    c = {"version": rd.symbol(st, False)}
    c["micro_version"] = rd.symbol(st, False)
    c["coder_type"] = rd.symbol(st, False)
    if c["coder_type"] == 2:
        raise ValueError("custom state tables are not restated")
    c["colorspace_type"] = rd.symbol(st, False)
    c["bits_per_raw_sample"] = rd.symbol(st, False)
    c["chroma_planes"] = rd.bit(st, 0)
    c["chroma_h_shift"] = rd.symbol(st, False)
    c["chroma_v_shift"] = rd.symbol(st, False)
    c["transparency"] = rd.bit(st, 0)
    c["num_h_slices"] = rd.symbol(st, False) + 1
    c["num_v_slices"] = rd.symbol(st, False) + 1
    n = rd.symbol(st, False)
    tables, counts = [], []
    for _ in range(n):
        count, qs = 1, []
        for _ in range(5):
            q, k = _read_quant_table(rd, count)
            qs.append(q)
            count *= k
        tables.append(qs)
        counts.append((count + 1) // 2)
    c["quant_tables"], c["context_count"] = tables, counts
    c["states_coded"] = [rd.bit(st, 0) for _ in range(n)]
    if any(c["states_coded"]):
        raise ValueError("coded initial states are not restated")
    c["ec"] = rd.symbol(st, False)
    c["intra"] = rd.symbol(st, False)
    return c


# ---- slices --------------------------------------------------------------------------------------------------------------


def _rct_planes(bgr):
    """JPEG2000-RCT of one slice: (G', B', R') int32 planes, G' = (B + R + 2G) >> 2, B' = B - G + 256, R' = R - G + 256."""
    b, g, r = (bgr[..., k].astype(np.int32) for k in range(3))
    bd, rd = b - g, r - g
    return [g + ((bd + rd) >> 2), bd + 256, rd + 256]


def _neighbours(p):
    """Per sample of plane p (h x w): L, T, LT, RT as libavcodec's two-line sample ring gives them. Above the first row
    every neighbour is 0; left of column 0, L is the sample above and LT the sample two rows up at column 0; right of the
    last column, RT repeats the last sample of the row above."""
    h, w = p.shape
    top = np.zeros((h, w + 2), np.int32)                  # row y holds row y - 1 with one guard column on each side
    top[1:, 1:w + 1] = p[:-1]
    top[1:, w + 1] = p[:-1, w - 1]
    top[2:, 0] = p[:-2, 0]
    T, LT, RT = top[:, 1:w + 1], top[:, 0:w], top[:, 2:w + 2]
    L = np.empty_like(p)
    L[:, 1:] = p[:, :-1]
    L[:, 0] = T[:, 0]
    return L, T, LT, RT


def _context_and_pred(p):
    L, T, LT, RT = _neighbours(p)
    ctx = QUANT11[(L - LT) & 0xFF] + 11 * QUANT11[(LT - T) & 0xFF] + 121 * QUANT11[(T - RT) & 0xFF]
    pred = np.median(np.stack([L, L + T - LT, T]), axis=0).astype(np.int32)
    return ctx, pred


def slice_symbols(bgr):
    """(context, folded residual) of every sample of one slice in coding order: rows top to bottom, per row G', then B',
    then R', left to right. Both arrays are (h, 3, w); contexts are >= 0 (a negative context flips the residual's sign);
    residuals are sign-extended from 9 bits, in [-256, 255]."""
    h, w = bgr.shape[:2]
    ctxs, res = np.empty((h, 3, w), np.int32), np.empty((h, 3, w), np.int32)
    for k, p in enumerate(_rct_planes(bgr)):
        ctx, pred = _context_and_pred(p)
        d = np.where(ctx < 0, pred - p, p - pred)
        ctxs[:, k], res[:, k] = np.abs(ctx), ((d + 256) & 511) - 256
    return ctxs, res


def _slice_header(rc, sx, sy):
    st = [128] * 32
    for v in (sx, sy, 0, 0, 0, 0, 3, 0, 0):    # slice_x, slice_y, width - 1, height - 1, two quant-table indices,
        rc.symbol(st, v, False)                # picture_structure 3 (progressive), sample aspect ratio 0:0


def encode_slice(bgr, sx, sy, rc=None):
    """One slice's bytes: its header, then every sample. `rc` continues an encoder (slice 0 after the keyframe bit)."""
    rc = rc or RangeEncoder()
    _slice_header(rc, sx, sy)
    ctxs, res = slice_symbols(bgr)
    states = [[[128] * 32 for _ in range(CONTEXT_COUNT)] for _ in range(2)]
    sym = rc.symbol
    for y in range(ctxs.shape[0]):
        for k in range(3):
            sp = states[1 if k else 0]
            for c, v in zip(ctxs[y, k].tolist(), res[y, k].tolist()):
                sym(sp[c], v, True)
    return rc.terminate()


def encode_frame(bgr, grid=None):
    """The packet of one BGR frame (H x W x 3 uint8): slices in raster order, each followed by its 24-bit size; slice 0
    starts with the keyframe bit on its own range coder."""
    h, w = bgr.shape[:2]
    nh, nv = grid or slice_grid(w, h)
    out = bytearray()
    for s, (x0, y0, x1, y1) in enumerate(slice_rects(w, h, (nh, nv))):
        rc = None
        if s == 0:
            rc = RangeEncoder()
            rc.bit([128], 0, 1)
        data = encode_slice(bgr[y0:y1, x0:x1], s % nh, s // nh, rc)
        out += data + len(data).to_bytes(3, "big")
    return bytes(out)


def split_slices(packet, trailer=3):
    """The slices of a version-3 packet as (start, size) in raster order, walked from the end by their 24-bit sizes."""
    out, end = [], len(packet)
    while end > 0:
        if end < trailer:
            raise ValueError("slice pointer chain broken")
        n = int.from_bytes(packet[end - trailer:end - trailer + 3], "big")
        if n + trailer > end:
            raise ValueError("slice pointer chain broken")
        out.append((end - trailer - n, n))
        end -= n + trailer
    return out[::-1]


def read_slice_header(rd):
    st = [128] * 32
    hdr = {k: rd.symbol(st, False) for k in ("slice_x", "slice_y", "slice_w_minus1", "slice_h_minus1")}
    return hdr, st


def decode_frame(packet, w, h, config):
    """BGR frame (H x W x 3 uint8) of a packet of this encoder's configuration. Raises on anything else, and checks that
    every slice ends exactly where libavcodec's decoder expects (it flags a slice whose coder stops short as damaged)."""
    if config["coder_type"] != 1 or config["transparency"] or config["colorspace_type"] != 1:
        raise ValueError("only the range-coded RGB configuration is decoded")
    nh, nv = config["num_h_slices"], config["num_v_slices"]
    q = config["quant_tables"]
    slices = split_slices(packet)
    if len(slices) != nh * nv:
        raise ValueError(f"{len(slices)} slices, the configuration has {nh * nv}")
    out = np.zeros((h, w, 3), np.uint8)
    for s, (start, size) in enumerate(slices):
        rd = RangeDecoder(packet[start:start + size + 3])           # libavcodec's coder may read into the trailer
        if s == 0 and not rd.bit([128], 0):
            raise ValueError("not a keyframe")
        hdr, st = read_slice_header(rd)
        qi = [rd.symbol(st, False) for _ in range(2)]
        ps, sar_n, sar_d = (rd.symbol(st, False) for _ in range(3))
        sx, sy = hdr["slice_x"], hdr["slice_y"]
        if hdr["slice_w_minus1"] or hdr["slice_h_minus1"] or ps != 3 or (sar_n, sar_d) != (0, 0):
            raise ValueError(f"unexpected slice header {hdr}")
        x0, x1 = w * sx // nh, w * (sx + 1) // nh
        y0, y1 = h * sy // nv, h * (sy + 1) // nv
        sw, sh = x1 - x0, y1 - y0
        tabs = [q[i] for i in qi]
        states = [[[128] * 32 for _ in range(config["context_count"][i])] for i in qi]
        planes = np.zeros((3, sh + 2, sw + 2), np.int32)            # one zero guard row on top, guard columns for L / RT
        for y in range(sh):
            for k in range(3):
                t = tabs[1 if k else 0]
                sp = states[1 if k else 0]
                P = planes[k]
                prev, cur = P[y], P[y + 1]
                cur[0] = prev[1]
                prev[sw + 1] = prev[sw]
                for x in range(1, sw + 1):
                    L, T, LT, RT = int(cur[x - 1]), int(prev[x]), int(prev[x - 1]), int(prev[x + 1])
                    ctx = int(t[0][(L - LT) & 0xFF] + t[1][(LT - T) & 0xFF] + t[2][(T - RT) & 0xFF])
                    d = rd.symbol(sp[abs(ctx)], True)
                    if ctx < 0:
                        d = -d
                    cur[x] = (sorted((L, L + T - LT, T))[1] + d) & 511
        # libavcodec decodes one more 0 with state 129 and flags the slice as damaged unless its coder then stands 2
        # bytes before the end of slice + trailer
        if rd.bit([129], 0) != 0 or rd.pos != size + 1:
            raise ValueError(f"slice {s}: bytestream end mismatch ({size + 1 - rd.pos} bytes)")
        g, b, r = (planes[k, 1:sh + 1, 1:sw + 1] for k in range(3))
        b, r = b - 256, r - 256
        g = g - ((b + r) >> 2)
        out[y0:y1, x0:x1] = np.stack([b + g, g, r + g], -1).astype(np.uint8)
    return out


# ---- Matroska ------------------------------------------------------------------------------------------------------------

EBML_MASTER = {0x1A45DFA3, 0x18538067, 0x1549A966, 0x1654AE6B, 0xAE, 0xE0, 0x1F43B675, 0xA0, 0x114D9B74, 0x4DBB,
               0x1C53BB6B, 0xBB, 0xB7, 0x1254C367, 0x7373, 0x63C0, 0x67C8}


def _vint(d, i, strip):
    b = d[i]
    n = 1
    while n <= 8 and not b & (0x80 >> (n - 1)):
        n += 1
    v = b & (0xFF >> n) if strip else b
    for k in range(1, n):
        v = (v << 8) | d[i + k]
    return v, i + n, (v == (1 << (7 * n)) - 1) if strip else False


def ebml_elements(d, i=0, end=None):
    """(id, payload start, payload end, children) for the elements of d[i:end]; masters are parsed recursively."""
    end = len(d) if end is None else end
    out = []
    while i < end:
        eid, i, _ = _vint(d, i, False)
        size, i, unknown = _vint(d, i, True)
        e = end if unknown else i + size
        out.append((eid, i, e, ebml_elements(d, i, e) if eid in EBML_MASTER else None))
        i = e
    return out


def _find(elems, eid):
    return [e for e in elems if e[0] == eid]


def read_mkv(path_or_bytes):
    """{"codec_id", "codec_private", "width", "height", "packets", "timestamps"} of the first video track of a
    Matroska file whose blocks are SimpleBlocks of track 1 without lacing."""
    d = path_or_bytes if isinstance(path_or_bytes, (bytes, bytearray)) else open(path_or_bytes, "rb").read()
    top = ebml_elements(d)
    seg = _find(top, 0x18538067)[0][3]
    track = _find(_find(seg, 0x1654AE6B)[0][3], 0xAE)[0]
    out = {"codec_id": None, "codec_private": b"", "width": 0, "height": 0, "packets": [], "timestamps": []}
    for eid, a, b, ch in track[3]:
        if eid == 0x86:
            out["codec_id"] = bytes(d[a:b]).decode()
        elif eid == 0x63A2:
            out["codec_private"] = bytes(d[a:b])
        elif eid == 0xE0:
            for vid, va, vb, _ in ch:
                if vid in (0xB0, 0xBA):
                    out["width" if vid == 0xB0 else "height"] = int.from_bytes(d[va:vb], "big")
    for _, _, _, cl in _find(seg, 0x1F43B675):
        tc = int.from_bytes(d[_find(cl, 0xE7)[0][1]:_find(cl, 0xE7)[0][2]], "big")
        for eid, a, b, _ in cl:
            if eid == 0xA3:
                _, j, _ = _vint(d, a, True)
                rel = int.from_bytes(d[j:j + 2], "big", signed=True)
                if d[j + 2] & 0x06:
                    raise ValueError("laced blocks are not read")
                out["packets"].append(bytes(d[j + 3:b]))
                out["timestamps"].append(tc + rel)
    return out
