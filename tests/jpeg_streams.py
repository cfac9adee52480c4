"""Deterministic JPEG streams with the header layouts other encoders write, for the JPEG decoder tests.

cv2.imencode always writes the same header: a JFIF APP0, component ids 1 2 3, Y on Huffman tables 0 and chroma on tables 1,
8-bit quantisation tables 0 and 1, one DQT / DHT segment per table.  Cameras, phones, image editors and libjpeg callers that
pick their own colour space write other headers.  The builders here start from a cv2 stream, split it into its header
segments and the data after the SOS header (entropy-coded data, EOI, whatever follows), and rewrite the header.  Every
rewrite keeps a stream that cv2.imdecode decodes, except the ones `error_streams` returns, which the decoders must refuse,
and a stream without its EOI: libjpeg warns about the premature end and cv2 gives up on some such streams and not on others,
so its expected output is the decode of the complete stream (the same whenever cv2 does decode both).

How cv2 (libjpeg-turbo, jdapimin.c default_decompress_parms) decides the colour space of a 3-component stream:
  1. a JFIF APP0 (payload >= 14 bytes starting "JFIF\\0") means YCbCr;
  2. else an Adobe APP14 (payload >= 12 bytes starting "Adobe") decides by its byte 11: 0 = RGB, 1 or anything else = YCbCr;
  3. else component ids 'R' 'G' 'B' mean RGB, any other ids YCbCr.
An RGB stream is upsampled as usual and written as (component 2, component 1, component 0).
"""
import struct

import numpy as np

SOI = b"\xff\xd8"
SOF0, SOF1, DHT, DQT, DRI, SOS, APP0, APP1, APP14, COM = 0xC0, 0xC1, 0xC4, 0xDB, 0xDD, 0xDA, 0xE0, 0xE1, 0xEE, 0xFE

def _cv2():
    import cv2
    return cv2


def sampling_flag(sampling):
    """'420' / '422' / '444' / '411' / '440' -> the cv2 IMWRITE_JPEG_SAMPLING_FACTOR_* value"""
    return getattr(_cv2(), "IMWRITE_JPEG_SAMPLING_FACTOR_" + sampling)


def encode(img, sampling="420", quality=90, rst=0, params=()):
    """cv2.imencode as bytes; rst > 0 adds a DRI of that many MCUs"""
    cv2 = _cv2()
    p = [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sampling_flag(sampling)] + list(params)
    if rst:
        p += [cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    ok, buf = cv2.imencode(".jpg", np.ascontiguousarray(img), p)
    assert ok
    return buf.tobytes()


def decode_cv2(stream):
    """cv2.imdecode(bytes, IMREAD_UNCHANGED), or None when cv2 cannot decode the stream"""
    cv2 = _cv2()
    return cv2.imdecode(np.frombuffer(stream, np.uint8), cv2.IMREAD_UNCHANGED)


# ---- segments --------------------------------------------------------------------------------------------------------------
def split(stream):
    """-> ([(marker, payload)] from SOI up to and including SOS, the bytes after the SOS header)"""
    assert stream[:2] == SOI
    segs, i = [], 2
    while True:
        assert stream[i] == 0xFF, "marker expected at %d" % i
        m = stream[i + 1]
        n = struct.unpack(">H", stream[i + 2:i + 4])[0]
        segs.append((m, stream[i + 4:i + 2 + n]))
        i += 2 + n
        if m == SOS:
            return segs, stream[i:]


def segment(m, payload, fill=0):
    return b"\xff" * fill + bytes([0xFF, m]) + struct.pack(">H", len(payload) + 2) + payload


def join(segs, tail, fill=0):
    """inverse of split; fill: 0xFF fill bytes before every header marker"""
    return SOI + b"".join(segment(m, p, fill) for m, p in segs) + tail


def parse_dqt(payload):
    """-> [(pq, tq, 64 values in zigzag order)]"""
    out, k = [], 0
    while k < len(payload):
        pq, tq = payload[k] >> 4, payload[k] & 15
        k += 1
        n = 128 if pq else 64
        vals = list(struct.unpack(">64H", payload[k:k + n])) if pq else list(payload[k:k + n])
        out.append((pq, tq, vals))
        k += n
    return out


def emit_dqt(tables):
    return b"".join(bytes([(pq << 4) | tq]) + (struct.pack(">64H", *v) if pq else bytes(v)) for pq, tq, v in tables)


def parse_dht(payload):
    """-> [(tc, th, bits[16], values)]"""
    out, k = [], 0
    while k < len(payload):
        tc, th = payload[k] >> 4, payload[k] & 15
        bits = list(payload[k + 1:k + 17])
        vals = bytes(payload[k + 17:k + 17 + sum(bits)])
        out.append((tc, th, bits, vals))
        k += 17 + sum(bits)
    return out


def emit_dht(tables):
    return b"".join(bytes([(tc << 4) | th] + list(bits)) + vals for tc, th, bits, vals in tables)


def _map(segs, m, fn):
    return [(mm, fn(p) if mm == m else p) for mm, p in segs]


def _sof_index(segs):
    return next(i for i, (m, _) in enumerate(segs) if m in (SOF0, SOF1))


# ---- rewrites --------------------------------------------------------------------------------------------------------------
def app0_jfif(payload_len=16):
    p = b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00" + bytes(max(0, payload_len - 14))
    return (APP0, p[:payload_len])


def app0_jfxx():
    return (APP0, b"JFXX\x00\x10" + bytes(8))


def app14_adobe(transform, payload_len=12):
    return (APP14, (b"Adobe" + struct.pack(">HHHB", 100, 0, 0, transform))[:payload_len])


def drop_app0(segs):
    return [(m, p) for m, p in segs if m != APP0]


def insert_after_soi(segs, *new):
    return list(new) + list(segs)


def set_component_ids(segs, ids):
    """SOF and SOS component ids"""
    def sof(p):
        p = bytearray(p)
        for c in range(3):
            p[6 + 3 * c] = ids[c]
        return bytes(p)

    def sos(p):
        p = bytearray(p)
        for c in range(3):
            p[1 + 2 * c] = ids[c]
        return bytes(p)
    return _map(_map(_map(segs, SOF0, sof), SOF1, sof), SOS, sos)


def swap_huffman(segs):
    """Y on DC/AC tables 1, chroma on tables 0"""
    def sos(p):
        p = bytearray(p)
        for c in range(3):
            p[2 + 2 * c] ^= 0x11
        return bytes(p)
    dht = _map(segs, DHT, lambda p: emit_dht([(tc, th ^ 1, b, v) for tc, th, b, v in parse_dht(p)]))
    return _map(dht, SOS, sos)


def requant_ids(segs, add=2):
    """quantisation tables 0/1 renumbered 2/3 (DQT and SOF)"""
    def sof(p):
        p = bytearray(p)
        for c in range(3):
            p[8 + 3 * c] += add
        return bytes(p)
    dqt = _map(segs, DQT, lambda p: emit_dqt([(pq, tq + add, v) for pq, tq, v in parse_dqt(p)]))
    return _map(dqt, SOF0, sof)


def dqt_16bit(segs):
    return _map(segs, DQT, lambda p: emit_dqt([(1, tq, v) for _, tq, v in parse_dqt(p)]))


def merge(segs, m):
    """every table of marker m in one segment, where the first one was"""
    body = b"".join(p for mm, p in segs if mm == m)
    out, done = [], False
    for mm, p in segs:
        if mm != m:
            out.append((mm, p))
        elif not done:
            out.append((m, body))
            done = True
    return out


def split_reversed(segs, m):
    """one segment per table, in reverse order (AC before DC, chroma before luma)"""
    parse, emit = (parse_dqt, emit_dqt) if m == DQT else (parse_dht, emit_dht)
    tables = [t for mm, p in segs if mm == m for t in parse(p)]
    out, done = [], False
    for mm, p in segs:
        if mm != m:
            out.append((mm, p))
        elif not done:
            out += [(m, emit([t])) for t in reversed(tables)]
            done = True
    return out


def define_twice(segs):
    """a different table 0 of each kind (DQT, DC, AC) first; the real definitions follow and win"""
    bogus_q = (0, 0, [1 + (i % 7) for i in range(64)])
    bogus_dc = (0, 0, [0, 1] + [0] * 14, bytes([7]))
    bogus_ac = (1, 0, [0, 2] + [0] * 14, bytes([0x01, 0x00]))
    return [(DQT, emit_dqt([bogus_q])), (DHT, emit_dht([bogus_dc, bogus_ac]))] + list(segs)


def move(segs, marker, where):
    """move the segments of `marker` to the start ('first') or behind the SOF ('after_sof')"""
    moved = [(m, p) for m, p in segs if m == marker]
    rest = [(m, p) for m, p in segs if m != marker]
    if where == "first":
        return moved + rest
    i = _sof_index(rest)
    return rest[:i + 1] + moved + rest[i + 1:]


def sof1(segs):
    return [(SOF1 if m == SOF0 else m, p) for m, p in segs]


def exif_orientation(value=6):
    tiff = b"MM\x00\x2a\x00\x00\x00\x08" + struct.pack(">H", 1) + struct.pack(">HHIHH", 0x0112, 3, 1, value, 0) + b"\x00\x00\x00\x00"
    return (APP1, b"Exif\x00\x00" + tiff)


def fill_in_scan(tail):
    """two 0xFF fill bytes before every marker of the entropy-coded data (RSTn and EOI)"""
    out, i = bytearray(), 0
    while i < len(tail):
        b = tail[i]
        if b == 0xFF and i + 1 < len(tail) and tail[i + 1] not in (0x00, 0xFF):
            out += b"\xff\xff"
        out.append(b)
        i += 1
    return bytes(out)


# ---- variant sets ----------------------------------------------------------------------------------------------------------
def colour_space_variants(img, sampling, quality=90, rst=0):
    """[(id, stream, rgb)]: the colour-space signalling of the module docstring; rgb = what cv2 decides"""
    segs, tail = split(encode(img, sampling, quality, rst))
    bare = drop_app0(segs)
    rgb_ids = set_component_ids(bare, b"RGB")
    v = [
        ("rgb-adobe0", join(insert_after_soi(bare, app14_adobe(0)), tail), True),
        ("rgb-ids", join(rgb_ids, tail), True),
        ("rgb-ids-adobe0", join(insert_after_soi(rgb_ids, app14_adobe(0)), tail), True),
        ("rgb-jfxx-adobe0", join(insert_after_soi(bare, app0_jfxx(), app14_adobe(0)), tail), True),
        ("rgb-shortjfif-adobe0", join(insert_after_soi(bare, app0_jfif(13), app14_adobe(0)), tail), True),
        ("rgb-adobe0-longer", join(insert_after_soi(bare, app14_adobe(0, 14)), tail), True),
        ("ycc-jfif-adobe0", join(segs[:1] + [app14_adobe(0)] + segs[1:], tail), False),
        ("ycc-adobe0-then-jfif", join(insert_after_soi(segs, app14_adobe(0)), tail), False),
        ("ycc-jfif-ids-rgb", join(set_component_ids(segs, b"RGB"), tail), False),
        ("ycc-adobe1", join(insert_after_soi(bare, app14_adobe(1)), tail), False),
        ("ycc-adobe2", join(insert_after_soi(bare, app14_adobe(2)), tail), False),
        ("ycc-adobe1-ids-rgb", join(insert_after_soi(rgb_ids, app14_adobe(1)), tail), False),
        ("ycc-adobe0-short", join(insert_after_soi(bare, app14_adobe(0, 11)), tail), False),
        ("ycc-no-markers", join(bare, tail), False),
        ("ycc-ids-012", join(set_component_ids(bare, bytes([0, 1, 2])), tail), False),
    ]
    return [("%s-%s-rst%d" % (name, sampling, rst), s, rgb) for name, s, rgb in v]


def layout_variants(img, sampling="420", quality=90, rst=0, seed=0):
    """[(id, stream, reference)]: tables, segment order and extras, stream end.  The expected output is
    cv2.imdecode(reference); reference is the stream itself except for the one without EOI."""
    base = encode(img, sampling, quality, rst)
    segs, tail = split(base)
    # a DRI for the orderings that move one: the stream's own, or a DRI of 0 (no restart markers)
    with_dri = segs if any(m == DRI for m, _ in segs) else segs[:_sof_index(segs)] + [(DRI, b"\x00\x00")] + segs[_sof_index(segs):]
    rng = np.random.default_rng(seed)
    second = encode(img[::2, ::2], "444", 70, rst=1)          # a complete JPEG with its own RSTn markers, as MPF / motion photos
    cv2 = _cv2()
    v = [
        ("huff-swapped", join(swap_huffman(segs), tail)),
        ("qt-ids-23", join(requant_ids(segs), tail)),
        ("tables-twice", join(define_twice(segs), tail)),
        ("dqt-dht-merged", join(merge(merge(segs, DQT), DHT), tail)),
        ("dqt-dht-split-reversed", join(split_reversed(split_reversed(merge(segs, DQT), DQT), DHT), tail)),
        ("dqt-16bit", join(dqt_16bit(segs), tail)),
        ("luma-chroma-quality", encode(img, sampling, quality, rst, [cv2.IMWRITE_JPEG_LUMA_QUALITY, 95, cv2.IMWRITE_JPEG_CHROMA_QUALITY, 40])),
        ("dri-first", join(move(with_dri, DRI, "first"), tail)),
        ("dqt-after-sof", join(move(segs, DQT, "after_sof"), tail)),
        ("sof1", join(sof1(segs), tail)),
        ("com", join(segs[:1] + [(COM, b"written by a test")] + segs[1:], tail)),
        ("exif-orientation-6", join(segs[:1] + [exif_orientation(6)] + segs[1:], tail)),
        ("fill-bytes", join(segs, tail, fill=2)),
        ("fill-bytes-in-scan", join(segs, fill_in_scan(tail))),
        ("trailing-random", base + rng.integers(0, 256, 3000, dtype=np.uint8).tobytes()),
        ("trailing-jpeg-rst", base + second),
        ("no-eoi", base[:-2], base),
    ]
    return [("%s-%s-rst%d" % (t[0], sampling, rst), t[1], t[-1]) for t in v]


def error_streams(img):
    """[(id, stream)] the decoders must refuse: 4:1:1, 4:4:0, SOF9 (arithmetic), a one-component scan, 12-bit precision"""
    segs, tail = split(encode(img, "420"))
    i = _sof_index(segs)

    def sof_byte0(p):
        return bytes([12]) + p[1:]

    def one_comp_sos(p):
        return bytes([1]) + p[1:3] + p[7:]
    return [
        ("sampling-411", encode(img, "411")),
        ("sampling-440", encode(img, "440")),
        ("sof9", join(segs[:i] + [(0xC9, segs[i][1])] + segs[i + 1:], tail)),
        ("sos-one-component", join(_map(segs, SOS, one_comp_sos), tail)),
        ("precision-12", join(_map(segs, SOF0, sof_byte0), tail)),
    ]


def tiny_streams(sizes=range(1, 34), samplings=("420", "422", "444"), rsts=(0, 1), seed=0):
    """[(id, stream)]: every (h, w) of sizes x sizes, noise content, with and without restart markers"""
    out = []
    for ss in samplings:
        for h in sizes:
            for w in sizes:
                img = np.random.default_rng(seed + 100 * h + w).integers(0, 256, (h, w, 3), dtype=np.uint8)
                for rst in rsts:
                    out.append(("tiny-%dx%d-%s-rst%d" % (h, w, ss, rst), encode(img, ss, 85, rst)))
    return out


def as_rgb(stream):
    """the same entropy-coded data tagged RGB (no JFIF, Adobe transform 0)"""
    segs, tail = split(stream)
    return join(insert_after_soi(drop_app0(segs), app14_adobe(0)), tail)
