/*
 * fd_jpeg_oracle.c — CPU restatement of the JPEG decode behind utils::byte_data_to_opencv (reference src/utils/utils.rs:8-52:
 * cv::imdecode(bytes, IMREAD_UNCHANGED) -> BGR Mat).  TEST INFRASTRUCTURE ONLY (see oracle/oracle.py); SURVEY 8(f) row N4.
 *
 * The algorithm lives in a third-party dependency that is absent from /root/reference: OpenCV (crate opencv = 0.92.0,
 * Cargo.lock:1175) -> its bundled libjpeg-turbo.  Restated from the published algorithms — ITU-T T.81 (marker syntax,
 * Huffman decoding Annex F.2.2) and libjpeg's decompressor with the defaults OpenCV leaves in place: dct_method = JDCT_ISLOW
 * (jidctint.c jpeg_idct_islow: 13-bit constants, PASS1_BITS 2), do_fancy_upsampling = TRUE (jdsample.c h2v2_fancy_upsample /
 * h2v1_fancy_upsample: triangle filter, context rows replicated at the image top and bottom, jdmainct.c), YCbCr -> BGR with the
 * 16-bit fixed-point tables of jdcolor.c.  Pinned against this container's cv2 4.13.0 (libjpeg-turbo 3.1.2, SIMD on):
 * bit-exact on every fixture of tests/test_oracle_vs_cv2.py::test_jpeg_* (4:2:0 / 4:2:2 / 4:4:4, odd sizes, restart intervals,
 * qualities 30..100) and on the committed golden vectors tests/golden/jpeg_golden.npz.
 *
 * Scope: baseline / extended-sequential 8-bit Huffman JPEG (SOF0 / SOF1), one interleaved scan, 3 components with luma
 * sampling 1x1, 2x1 or 2x2 and 1x1 chroma (4:4:4, 4:2:2, 4:2:0), YCbCr or RGB as libjpeg's default_decompress_parms
 * decides it (JFIF APP0, else the Adobe APP14 transform, else component ids 'R' 'G' 'B'); an RGB stream is upsampled the same
 * way and written as (comp 2, comp 1, comp 0).  4:1:1, 4:4:0, non-interleaved, progressive, arithmetic, 12-bit, grayscale and
 * CMYK streams return an error code.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define FDO_API __attribute__((visibility("default")))

enum { FDJ_OK = 0, FDJ_ERR_SYNTAX = -1, FDJ_ERR_UNSUPPORTED = -2, FDJ_ERR_TRUNCATED = -3 };

static const uint8_t ZIGZAG[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                   41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                   30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

typedef struct {
    int present;
    uint8_t bits[17], vals[256];
    int mincode[17], maxcode[18], valptr[17];   /* T.81 F.2.2.3 decoding tables */
} huff_t;

typedef struct {
    int h, w, ncomp, restart;
    int id[3], hs[3], vs[3], tq[3], td[3], ta[3];
    int jfif, adobe, adobe_transform;   /* JFIF APP0 seen, Adobe APP14 seen and its transform byte */
    int rgb;                            /* the components are R, G, B (no colour conversion) */
    uint16_t qt[4][64];   /* natural (row-major) order */
    int qt_present[4];
    huff_t dc[4], ac[4];
    const uint8_t *scan;  /* entropy-coded segment */
    size_t scan_len;
} jpeg_t;

static void build_huff(huff_t *t) {   /* T.81 C.2 + F.2.2.3 */
    int code = 0, k = 0;
    for (int l = 1; l <= 16; ++l) {
        t->valptr[l] = k;
        t->mincode[l] = code;
        code += t->bits[l];
        k += t->bits[l];
        t->maxcode[l] = t->bits[l] ? code - 1 : -1;
        code <<= 1;
    }
    t->maxcode[17] = 0x7fffffff;
    t->present = 1;
}

static int parse(const uint8_t *p, size_t n, jpeg_t *j) {
    memset(j, 0, sizeof(*j));
    if (n < 4 || p[0] != 0xFF || p[1] != 0xD8) return FDJ_ERR_SYNTAX;
    size_t i = 2;
    int have_sof = 0;
    while (i + 4 <= n) {
        if (p[i] != 0xFF) return FDJ_ERR_SYNTAX;
        while (i < n && p[i] == 0xFF) ++i;          /* fill bytes */
        if (i >= n) return FDJ_ERR_TRUNCATED;
        const int m = p[i++];
        if (m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) continue;
        if (m == 0xD9) return FDJ_ERR_SYNTAX;       /* EOI before SOS */
        if (i + 2 > n) return FDJ_ERR_TRUNCATED;
        const size_t len = ((size_t)p[i] << 8) | p[i + 1];
        if (len < 2 || i + len > n) return FDJ_ERR_TRUNCATED;
        const uint8_t *s = p + i + 2;
        const size_t sl = len - 2;
        if (m == 0xDB) {                            /* DQT */
            size_t k = 0;
            while (k < sl) {
                const int pq = s[k] >> 4, tq = s[k] & 15;
                ++k;
                if (tq > 3 || k + (pq ? 128 : 64) > sl) return FDJ_ERR_SYNTAX;
                for (int z = 0; z < 64; ++z) {
                    const int v = pq ? ((s[k] << 8) | s[k + 1]) : s[k];
                    k += pq ? 2 : 1;
                    j->qt[tq][ZIGZAG[z]] = (uint16_t)v;
                }
                j->qt_present[tq] = 1;
            }
        } else if (m == 0xC4) {                     /* DHT */
            size_t k = 0;
            while (k < sl) {
                const int tc = s[k] >> 4, th = s[k] & 15;
                ++k;
                if (tc > 1 || th > 3 || k + 16 > sl) return FDJ_ERR_SYNTAX;
                huff_t *t = tc ? &j->ac[th] : &j->dc[th];
                int total = 0;
                t->bits[0] = 0;
                for (int l = 1; l <= 16; ++l) { t->bits[l] = s[k++]; total += t->bits[l]; }
                if (total > 256 || k + (size_t)total > sl) return FDJ_ERR_SYNTAX;
                memcpy(t->vals, s + k, (size_t)total);
                k += (size_t)total;
                build_huff(t);
            }
        } else if (m == 0xC0 || m == 0xC1) {        /* SOF0 / SOF1 */
            if (sl < 6 || s[0] != 8) return FDJ_ERR_UNSUPPORTED;
            j->h = (s[1] << 8) | s[2];
            j->w = (s[3] << 8) | s[4];
            j->ncomp = s[5];
            if (j->ncomp != 3 || sl < 6 + 9 || j->h == 0 || j->w == 0) return FDJ_ERR_UNSUPPORTED;
            for (int c = 0; c < 3; ++c) {
                j->id[c] = s[6 + 3 * c];
                j->hs[c] = s[7 + 3 * c] >> 4;
                j->vs[c] = s[7 + 3 * c] & 15;
                j->tq[c] = s[8 + 3 * c];
                if (j->tq[c] > 3) return FDJ_ERR_SYNTAX;
            }
            if (j->hs[1] != 1 || j->vs[1] != 1 || j->hs[2] != 1 || j->vs[2] != 1) return FDJ_ERR_UNSUPPORTED;
            if (!((j->hs[0] == 1 && j->vs[0] == 1) || (j->hs[0] == 2 && j->vs[0] == 1) || (j->hs[0] == 2 && j->vs[0] == 2)))
                return FDJ_ERR_UNSUPPORTED;
            have_sof = 1;
        } else if (m >= 0xC2 && m <= 0xCF && m != 0xC4 && m != 0xC8 && m != 0xCC) {
            return FDJ_ERR_UNSUPPORTED;             /* progressive, lossless, arithmetic, hierarchical */
        } else if (m == 0xE0) {                     /* APP0: JFIF (jdmarker.c examine_app0: >= 14 bytes, "JFIF\0") */
            if (sl >= 14 && !memcmp(s, "JFIF", 5)) j->jfif = 1;
        } else if (m == 0xEE) {                     /* APP14: Adobe (examine_app14: >= 12 bytes, "Adobe"), byte 11 = transform */
            if (sl >= 12 && !memcmp(s, "Adobe", 5)) { j->adobe = 1; j->adobe_transform = s[11]; }
        } else if (m == 0xDD) {                     /* DRI */
            if (sl < 2) return FDJ_ERR_SYNTAX;
            j->restart = (s[0] << 8) | s[1];
        } else if (m == 0xDA) {                     /* SOS */
            if (!have_sof || sl < 1 || s[0] != 3 || sl < 1 + 6 + 3) return FDJ_ERR_UNSUPPORTED;
            for (int c = 0; c < 3; ++c) {
                if (s[1 + 2 * c] != j->id[c]) return FDJ_ERR_UNSUPPORTED;
                j->td[c] = s[2 + 2 * c] >> 4;
                j->ta[c] = s[2 + 2 * c] & 15;
                if (j->td[c] > 3 || j->ta[c] > 3 || !j->dc[j->td[c]].present || !j->ac[j->ta[c]].present || !j->qt_present[j->tq[c]])
                    return FDJ_ERR_SYNTAX;
            }
            if (s[7] != 0 || s[8] != 63) return FDJ_ERR_UNSUPPORTED;
            /* jdapimin.c default_decompress_parms, 3 components: JFIF means YCbCr; else an Adobe transform of 0 means RGB (any
             * other transform YCbCr); else component ids 'R' 'G' 'B' mean RGB, any others YCbCr */
            if (j->jfif) j->rgb = 0;
            else if (j->adobe) j->rgb = j->adobe_transform == 0;
            else j->rgb = j->id[0] == 'R' && j->id[1] == 'G' && j->id[2] == 'B';
            j->scan = p + i + len;
            j->scan_len = n - (i + len);
            return FDJ_OK;
        }
        i += len;
    }
    return FDJ_ERR_TRUNCATED;
}

/* bit reader over the entropy-coded segment: FF00 -> FF, stops (zero fill) at any other marker */
typedef struct {
    const uint8_t *p;
    size_t n, i;
    uint32_t acc;
    int cnt, hit_marker;
} bits_t;

static void fill(bits_t *b) {
    while (b->cnt <= 24) {
        int byte = 0;
        if (!b->hit_marker && b->i < b->n) {
            byte = b->p[b->i];
            if (byte == 0xFF) {
                if (b->i + 1 < b->n && b->p[b->i + 1] == 0x00) b->i += 2;
                else { b->hit_marker = 1; byte = 0; }
            } else {
                b->i += 1;
            }
        }
        b->acc |= (uint32_t)byte << (24 - b->cnt);
        b->cnt += 8;
    }
}
static int getbits(bits_t *b, int n) {
    if (n == 0) return 0;
    fill(b);
    const int v = (int)(b->acc >> (32 - n));
    b->acc <<= n;
    b->cnt -= n;
    return v;
}
static int decode_sym(bits_t *b, const huff_t *t) {   /* F.2.2.3 DECODE */
    int code = getbits(b, 1), l = 1;
    while (l <= 16 && code > t->maxcode[l]) {
        code = (code << 1) | getbits(b, 1);
        ++l;
    }
    if (l > 16) return 0;
    return t->vals[t->valptr[l] + code - t->mincode[l]];
}
static int extend(int v, int s) { return v < (1 << (s - 1)) ? v - (1 << s) + 1 : v; }   /* F.2.2.1 EXTEND */

/* ---- jidctint.c jpeg_idct_islow, with the dequantisation it performs ------------------------------------------------------ */
#define CONST_BITS 13
#define PASS1_BITS 2
#define DESCALE(x, n) (((x) + ((int32_t)1 << ((n) - 1))) >> (n))
static inline uint8_t range_limit(int32_t x) {   /* sample_range_limit + CENTERJSAMPLE indexed with (x & RANGE_MASK) */
    const int m = x & 1023;
    return (uint8_t)(m < 128 ? m + 128 : (m < 512 ? 255 : (m < 896 ? 0 : m - 896)));
}
static void idct_islow(const int16_t *in, const uint16_t *q, uint8_t *out, int out_pitch) {
    int32_t ws[64];
    for (int c = 0; c < 8; ++c) {
        const int16_t *i = in + c;
        const uint16_t *qq = q + c;
        int32_t *w = ws + c;
        if (!i[8] && !i[16] && !i[24] && !i[32] && !i[40] && !i[48] && !i[56]) {
            const int32_t dc = (int32_t)(i[0] * qq[0]) << PASS1_BITS;
            for (int k = 0; k < 8; ++k) w[8 * k] = dc;
            continue;
        }
        int32_t z2 = i[16] * qq[16], z3 = i[48] * qq[48];
        int32_t z1 = (z2 + z3) * 4433;
        int32_t tmp2 = z1 + z3 * (-15137), tmp3 = z1 + z2 * 6270;
        z2 = i[0] * qq[0];
        z3 = i[32] * qq[32];
        int32_t tmp0 = (z2 + z3) << CONST_BITS, tmp1 = (z2 - z3) << CONST_BITS;
        const int32_t tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
        tmp0 = i[56] * qq[56];
        tmp1 = i[40] * qq[40];
        tmp2 = i[24] * qq[24];
        tmp3 = i[8] * qq[8];
        z1 = tmp0 + tmp3;
        z2 = tmp1 + tmp2;
        z3 = tmp0 + tmp2;
        int32_t z4 = tmp1 + tmp3;
        const int32_t z5 = (z3 + z4) * 9633;
        tmp0 *= 2446; tmp1 *= 16819; tmp2 *= 25172; tmp3 *= 12299;
        z1 *= -7373; z2 *= -20995; z3 *= -16069; z4 *= -3196;
        z3 += z5;
        z4 += z5;
        tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
        w[0] = DESCALE(tmp10 + tmp3, CONST_BITS - PASS1_BITS);
        w[56] = DESCALE(tmp10 - tmp3, CONST_BITS - PASS1_BITS);
        w[8] = DESCALE(tmp11 + tmp2, CONST_BITS - PASS1_BITS);
        w[48] = DESCALE(tmp11 - tmp2, CONST_BITS - PASS1_BITS);
        w[16] = DESCALE(tmp12 + tmp1, CONST_BITS - PASS1_BITS);
        w[40] = DESCALE(tmp12 - tmp1, CONST_BITS - PASS1_BITS);
        w[24] = DESCALE(tmp13 + tmp0, CONST_BITS - PASS1_BITS);
        w[32] = DESCALE(tmp13 - tmp0, CONST_BITS - PASS1_BITS);
    }
    for (int r = 0; r < 8; ++r) {
        const int32_t *w = ws + 8 * r;
        uint8_t *o = out + (size_t)r * out_pitch;
        int32_t z2 = w[2], z3 = w[6];
        int32_t z1 = (z2 + z3) * 4433;
        int32_t tmp2 = z1 + z3 * (-15137), tmp3 = z1 + z2 * 6270;
        int32_t tmp0 = (w[0] + w[4]) << CONST_BITS, tmp1 = (w[0] - w[4]) << CONST_BITS;
        const int32_t tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
        tmp0 = w[7]; tmp1 = w[5]; tmp2 = w[3]; tmp3 = w[1];
        z1 = tmp0 + tmp3;
        z2 = tmp1 + tmp2;
        z3 = tmp0 + tmp2;
        int32_t z4 = tmp1 + tmp3;
        const int32_t z5 = (z3 + z4) * 9633;
        tmp0 *= 2446; tmp1 *= 16819; tmp2 *= 25172; tmp3 *= 12299;
        z1 *= -7373; z2 *= -20995; z3 *= -16069; z4 *= -3196;
        z3 += z5;
        z4 += z5;
        tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
        o[0] = range_limit(DESCALE(tmp10 + tmp3, CONST_BITS + PASS1_BITS + 3));
        o[7] = range_limit(DESCALE(tmp10 - tmp3, CONST_BITS + PASS1_BITS + 3));
        o[1] = range_limit(DESCALE(tmp11 + tmp2, CONST_BITS + PASS1_BITS + 3));
        o[6] = range_limit(DESCALE(tmp11 - tmp2, CONST_BITS + PASS1_BITS + 3));
        o[2] = range_limit(DESCALE(tmp12 + tmp1, CONST_BITS + PASS1_BITS + 3));
        o[5] = range_limit(DESCALE(tmp12 - tmp1, CONST_BITS + PASS1_BITS + 3));
        o[3] = range_limit(DESCALE(tmp13 + tmp0, CONST_BITS + PASS1_BITS + 3));
        o[4] = range_limit(DESCALE(tmp13 - tmp0, CONST_BITS + PASS1_BITS + 3));
    }
}

/* chroma sample at full resolution: jdsample.c fullsize / h2v1_fancy / h2v2_fancy with jdmainct.c's replicated context rows */
static inline int chroma_at(const uint8_t *pl, int pitch, int dw, int dh, int hs, int vs, int x, int y) {
    if (hs == 1 && vs == 1) return pl[(size_t)y * pitch + x];
    const int cx = x >> 1;
    /* jdsample.c jinit_upsampler: the fancy (triangle) filters are selected only when downsampled_width > 2; narrower
     * components take h2v1_upsample / h2v2_upsample (pixel replication) */
    if (dw <= 2) return pl[(size_t)(vs == 2 ? y >> 1 : y) * pitch + cx];
    if (vs == 1) {   /* h2v1_fancy_upsample */
        const uint8_t *r = pl + (size_t)y * pitch;
        const int v = r[cx];
        if (!(x & 1)) return cx == 0 ? v : (v * 3 + r[cx - 1] + 1) >> 2;
        if (cx == 0) return (v * 3 + r[1] + 2) >> 2;
        return cx == dw - 1 ? v : (v * 3 + r[cx + 1] + 2) >> 2;
    }
    /* h2v2_fancy_upsample: nearest row cy, next nearest above (even y) or below (odd y), clamped to the real rows */
    const int cy = y >> 1;
    int ny = (y & 1) ? cy + 1 : cy - 1;
    ny = ny < 0 ? 0 : (ny > dh - 1 ? dh - 1 : ny);
    const uint8_t *r0 = pl + (size_t)cy * pitch, *r1 = pl + (size_t)ny * pitch;
    const int t = r0[cx] * 3 + r1[cx];
    if (cx == 0) return (x & 1) ? (t * 3 + (r0[1] * 3 + r1[1]) + 7) >> 4 : (t * 4 + 8) >> 4;
    if (!(x & 1)) return (t * 3 + (r0[cx - 1] * 3 + r1[cx - 1]) + 8) >> 4;
    return cx == dw - 1 ? (t * 4 + 7) >> 4 : (t * 3 + (r0[cx + 1] * 3 + r1[cx + 1]) + 7) >> 4;
}

static inline uint8_t clamp8(int v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

FDO_API int fdo_jpeg_info(const uint8_t *jpeg, size_t n, int *h, int *w, int *subsampling) {
    jpeg_t j;
    const int rc = parse(jpeg, n, &j);
    if (rc != FDJ_OK) return rc;
    *h = j.h;
    *w = j.w;
    if (subsampling) *subsampling = j.hs[0] * 10 + j.vs[0];   /* 11 = 4:4:4, 21 = 4:2:2, 22 = 4:2:0 */
    return FDJ_OK;
}

/* out: h x w x 3 BGR (pitch bytes per row).  Returns FDJ_OK or a negative error. */
FDO_API int fdo_jpeg_decode_bgr(const uint8_t *jpeg, size_t n, uint8_t *out, int pitch) {
    jpeg_t j;
    int rc = parse(jpeg, n, &j);
    if (rc != FDJ_OK) return rc;
    const int H = j.hs[0], V = j.vs[0];
    const int mcux = (j.w + 8 * H - 1) / (8 * H), mcuy = (j.h + 8 * V - 1) / (8 * V);
    int pw[3], ph[3];
    uint8_t *plane[3];
    for (int c = 0; c < 3; ++c) {
        pw[c] = mcux * j.hs[c] * 8;
        ph[c] = mcuy * j.vs[c] * 8;
        plane[c] = (uint8_t *)malloc((size_t)pw[c] * ph[c] + 16);
    }
    bits_t b;
    memset(&b, 0, sizeof(b));
    b.p = j.scan;
    b.n = j.scan_len;
    int pred[3] = {0, 0, 0};
    int16_t coef[64];
    int mcu_count = 0;
    for (int my = 0; my < mcuy; ++my)
        for (int mx = 0; mx < mcux; ++mx) {
            if (j.restart && mcu_count && mcu_count % j.restart == 0) {   /* RSTn: byte-align, skip the marker, reset DC */
                b.acc = 0;
                b.cnt = 0;
                if (b.hit_marker) {
                    while (b.i + 1 < b.n && !(b.p[b.i] == 0xFF && b.p[b.i + 1] >= 0xD0 && b.p[b.i + 1] <= 0xD7)) ++b.i;
                    b.i += 2;
                    b.hit_marker = 0;
                } else if (b.i + 1 < b.n && b.p[b.i] == 0xFF && b.p[b.i + 1] >= 0xD0 && b.p[b.i + 1] <= 0xD7) {
                    b.i += 2;
                }
                pred[0] = pred[1] = pred[2] = 0;
            }
            ++mcu_count;
            for (int c = 0; c < 3; ++c)
                for (int v = 0; v < j.vs[c]; ++v)
                    for (int hh = 0; hh < j.hs[c]; ++hh) {
                        memset(coef, 0, sizeof(coef));
                        int s = decode_sym(&b, &j.dc[j.td[c]]);
                        if (s) pred[c] += extend(getbits(&b, s), s);
                        coef[0] = (int16_t)pred[c];
                        for (int k = 1; k < 64;) {
                            const int rs = decode_sym(&b, &j.ac[j.ta[c]]);
                            const int r = rs >> 4;
                            s = rs & 15;
                            if (s == 0) {
                                if (r != 15) break;
                                k += 16;
                                continue;
                            }
                            k += r;
                            if (k > 63) break;
                            coef[ZIGZAG[k]] = (int16_t)extend(getbits(&b, s), s);
                            ++k;
                        }
                        const int bx = mx * j.hs[c] + hh, by = my * j.vs[c] + v;
                        idct_islow(coef, j.qt[j.tq[c]], plane[c] + (size_t)by * 8 * pw[c] + (size_t)bx * 8, pw[c]);
                    }
        }
    /* jdcolor.c build_ycc_rgb_table + ycc_rgb_convert (JCS_EXT_BGR ordering); an RGB stream takes rgb_rgb_convert: the
     * upsampled components are only reordered */
    const int dw = (j.w * 1 + H - 1) / H, dh = (j.h * 1 + V - 1) / V;   /* downsampled_width / _height of the chroma components */
    for (int y = 0; y < j.h; ++y) {
        uint8_t *o = out + (size_t)y * pitch;
        for (int x = 0; x < j.w; ++x) {
            const int Y = plane[0][(size_t)y * pw[0] + x];
            const int cb = chroma_at(plane[1], pw[1], dw, dh, H, V, x, y) - 128;
            const int cr = chroma_at(plane[2], pw[2], dw, dh, H, V, x, y) - 128;
            if (j.rgb) {
                o[3 * x] = (uint8_t)(cr + 128);
                o[3 * x + 1] = (uint8_t)(cb + 128);
                o[3 * x + 2] = (uint8_t)Y;
                continue;
            }
            const int r = Y + (int)((91881 * cr + 32768) >> 16);                         /* FIX(1.40200) */
            const int g = Y + (int)(((-22554) * cb + 32768 + (-46802) * cr) >> 16);      /* -FIX(0.34414), -FIX(0.71414) */
            const int bl = Y + (int)((116130 * cb + 32768) >> 16);                       /* FIX(1.77200) */
            o[3 * x] = clamp8(bl);
            o[3 * x + 1] = clamp8(g);
            o[3 * x + 2] = clamp8(r);
        }
    }
    for (int c = 0; c < 3; ++c) free(plane[c]);
    return FDJ_OK;
}
