// fd_jpeg.cu — SURVEY 8(f) row N4: utils::byte_data_to_opencv (reference src/utils/utils.rs:8-52 = cv::imdecode(bytes,
// IMREAD_UNCHANGED)) for baseline JPEG, producing DEVICE-resident BGR frames for fd_preprocess_batch / fd_align_*.
//
// Split of the work:
//   entropy decoding (ITU-T T.81 Annex F.2.2).  An entropy-coded segment is a serial bit stream: every symbol's position
//          depends on all earlier ones, and the only synchronisation points the format has are restart markers (DRI / RSTn).
//          * streams WITH restart markers less than 32 MCUs apart: the device locates the markers (jpeg_iv_write_kernel); the compressed bytes go to the
//            device as they are and `jpeg_huffman_kernel` decodes one restart interval per thread (Huffman lookup tables in
//            shared memory, coefficients written straight into the device coefficient blocks) — the 1.3 MB stream of a 1080p
//            frame is all that crosses PCIe;
//          * streams WITHOUT restart markers (what most encoders emit by default) and streams with LONG restart intervals (too
//            few intervals for one thread each; the markers become boundaries of the chain) are copied as they are too, unstuffed on the
//            device (jpeg_unstuff_*_kernel) and decoded by self-synchronising sub-sequences: jpeg_sync_kernel rounds to the
//            fixed point of the chain of decoder states, then jpeg_write_kernel + jpeg_dc_kernel (see the section below);
//          * a host Huffman decoder (one image per worker thread, pinned coefficient blocks, copied) remains for streams with
//            more than two DC / AC tables or an inconsistent marker sequence, and behind FD_JPEG_HOST_HUFFMAN /
//            FD_JPEG_NO_SELFSYNC for A/B runs;
//          both device decoders assemble blocks in shared memory and write them out whole, in SCAN order (stage_flush);
//   device `jpeg_idct_kernel`: dequantisation + libjpeg's jpeg_idct_islow (jidctint.c: 13-bit constants, PASS1_BITS 2, the
//          range-limit table with its wrap-around), 8 threads per block;
//          `jpeg_color_kernel`: chroma upsampling (jdsample.c h2v1 / h2v2 "fancy" triangle filters with jdmainct.c's replicated
//          context rows; plain replication when downsampled_width <= 2, as jinit_upsampler selects) + YCbCr -> BGR with
//          jdcolor.c's 16-bit fixed-point constants, 8 pixels per thread sharing the filter's column sums.  A stream whose
//          components are R, G, B (see JpegHeader::rgb) is upsampled the same way and only reordered (jdcolor.c rgb_rgb_convert).
// Every integer operation follows libjpeg-turbo's decompressor with the defaults OpenCV leaves in place (JDCT_ISLOW,
// do_fancy_upsampling), so the frames are bit-identical to cv2.imdecode (tests/test_gpu_jpeg.py, golden vectors from cv2 4.13).
// Scope: SOF0 / SOF1 8-bit, one interleaved 3-component scan, 4:4:4 / 4:2:2 / 4:2:0, DRI/RSTn, YCbCr or RGB components (as
// libjpeg decides: JFIF APP0, else the Adobe APP14 transform, else component ids 'R' 'G' 'B').  4:1:1, 4:4:0, non-interleaved,
// progressive, arithmetic, 12-bit, grayscale and CMYK streams return FD_ERR_INVALID (the reference would hand them to OpenCV).
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <thread>
#include <vector>
#include "fd_internal.cuh"

namespace fd {

static const uint8_t JZIGZAG[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                    41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                    30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

constexpr int HUFF_LOOKAHEAD = 10;

struct HuffTable {
    bool present = false;
    uint8_t bits[17] = {0}, vals[256] = {0};
    int maxcode[18], mincode[17], valptr[17];
    unsigned maxleft[17];                 // first 16-bit left-aligned code value that is LONGER than l bits (non-decreasing in l)
    uint16_t look[1 << HUFF_LOOKAHEAD];   // (length << 8) | symbol for codes of <= HUFF_LOOKAHEAD bits, 0 = longer code
    void build() {
        int code = 0, k = 0;
        memset(look, 0, sizeof(look));
        for (int l = 1; l <= 16; ++l) {
            valptr[l] = k;
            mincode[l] = code;
            for (int i = 0; i < bits[l]; ++i, ++k, ++code) {
                if (l <= HUFF_LOOKAHEAD) {
                    const int first = code << (HUFF_LOOKAHEAD - l), n = 1 << (HUFF_LOOKAHEAD - l);
                    for (int j = 0; j < n; ++j) look[first + j] = (uint16_t)((l << 8) | vals[k]);
                }
            }
            maxcode[l] = bits[l] ? code - 1 : -1;
            maxleft[l] = (unsigned)code << (16 - l);
            code <<= 1;
        }
        maxleft[0] = 0;
        maxcode[17] = 0x7fffffff;
        present = true;
    }
};

// Huffman tables of one image as the device decoder wants them (baseline: at most 2 DC + 2 AC tables)
struct JpegHuffDev {
    uint16_t look[4][1 << HUFF_LOOKAHEAD];   // [0,1] DC tables 0/1, [2,3] AC tables 0/1
    int mincode[4][17], valptr[4][17];
    unsigned maxleft[4][17];
    uint8_t vals[4][256];
};

struct JpegHeader {
    int h = 0, w = 0, restart = 0;
    int id[3], hs[3], vs[3], tq[3], td[3], ta[3];
    bool jfif = false, adobe = false;   // a JFIF APP0 / an Adobe APP14 was seen (jdmarker.c examine_app0 / examine_app14)
    int adobe_transform = 0;
    bool rgb = false;                   // the components are R, G, B: no colour conversion (jdapimin.c default_decompress_parms)
    uint16_t qt[4][64];
    bool qt_present[4] = {false, false, false, false};
    HuffTable dc[4], ac[4];
    const uint8_t *scan = nullptr;
    size_t scan_len = 0;
    // derived geometry
    int mcux = 0, mcuy = 0;
    int pw[3], ph[3];          // component plane sizes (multiples of 8 x the MCU grid)
    size_t blocks[3];          // DCT blocks per component
};

static const char *parse_jpeg(const uint8_t *p, size_t n, JpegHeader *j) {
    if (!p || n < 4 || p[0] != 0xFF || p[1] != 0xD8) return "not a JPEG stream (no SOI)";
    size_t i = 2;
    bool have_sof = false;
    while (i + 4 <= n) {
        if (p[i] != 0xFF) return "marker expected";
        while (i < n && p[i] == 0xFF) ++i;
        if (i >= n) break;
        const int m = p[i++];
        if (m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) continue;
        if (m == 0xD9) return "EOI before SOS";
        if (i + 2 > n) break;
        const size_t len = ((size_t)p[i] << 8) | p[i + 1];
        if (len < 2 || i + len > n) break;
        const uint8_t *s = p + i + 2;
        const size_t sl = len - 2;
        switch (m) {
            case 0xDB: {
                size_t k = 0;
                while (k < sl) {
                    const int pq = s[k] >> 4, tq = s[k] & 15;
                    ++k;
                    if (tq > 3 || k + (pq ? 128u : 64u) > sl) return "bad DQT";
                    for (int z = 0; z < 64; ++z) {
                        j->qt[tq][JZIGZAG[z]] = (uint16_t)(pq ? ((s[k] << 8) | s[k + 1]) : s[k]);
                        k += pq ? 2 : 1;
                    }
                    j->qt_present[tq] = true;
                }
                break;
            }
            case 0xC4: {
                size_t k = 0;
                while (k < sl) {
                    const int tc = s[k] >> 4, th = s[k] & 15;
                    ++k;
                    if (tc > 1 || th > 3 || k + 16 > sl) return "bad DHT";
                    HuffTable &t = tc ? j->ac[th] : j->dc[th];
                    int total = 0;
                    for (int l = 1; l <= 16; ++l) { t.bits[l] = s[k++]; total += t.bits[l]; }
                    if (total > 256 || k + (size_t)total > sl) return "bad DHT";
                    memcpy(t.vals, s + k, (size_t)total);
                    k += (size_t)total;
                    t.build();
                }
                break;
            }
            case 0xC0:
            case 0xC1: {
                if (sl < 15 || s[0] != 8) return "unsupported sample precision";
                j->h = (s[1] << 8) | s[2];
                j->w = (s[3] << 8) | s[4];
                if (s[5] != 3) return "unsupported component count (grayscale / CMYK)";
                if (j->h == 0 || j->w == 0) return "empty image";
                for (int c = 0; c < 3; ++c) {
                    j->id[c] = s[6 + 3 * c];
                    j->hs[c] = s[7 + 3 * c] >> 4;
                    j->vs[c] = s[7 + 3 * c] & 15;
                    j->tq[c] = s[8 + 3 * c];
                    if (j->tq[c] > 3) return "bad SOF";
                }
                if (j->hs[1] != 1 || j->vs[1] != 1 || j->hs[2] != 1 || j->vs[2] != 1) return "unsupported chroma sampling";
                if (!((j->hs[0] == 1 && j->vs[0] == 1) || (j->hs[0] == 2 && j->vs[0] == 1) || (j->hs[0] == 2 && j->vs[0] == 2)))
                    return "unsupported luma sampling (4:4:4, 4:2:2 and 4:2:0 are)";
                have_sof = true;
                break;
            }
            case 0xE0:   // JFIF: payload >= 14 bytes starting "JFIF\0"
                if (sl >= 14 && !memcmp(s, "JFIF", 5)) j->jfif = true;
                break;
            case 0xEE:   // Adobe: payload >= 12 bytes starting "Adobe"; byte 11 is the colour transform
                if (sl >= 12 && !memcmp(s, "Adobe", 5)) { j->adobe = true; j->adobe_transform = s[11]; }
                break;
            case 0xDD:
                if (sl < 2) return "bad DRI";
                j->restart = (s[0] << 8) | s[1];
                break;
            case 0xDA: {
                if (!have_sof) return "SOS before SOF";
                if (sl < 10 || s[0] != 3) return "unsupported scan (one interleaved 3-component scan is)";
                for (int c = 0; c < 3; ++c) {
                    if (s[1 + 2 * c] != j->id[c]) return "unsupported scan component order";
                    j->td[c] = s[2 + 2 * c] >> 4;
                    j->ta[c] = s[2 + 2 * c] & 15;
                    if (j->td[c] > 3 || j->ta[c] > 3 || !j->dc[j->td[c]].present || !j->ac[j->ta[c]].present || !j->qt_present[j->tq[c]])
                        return "scan refers to a missing table";
                }
                if (s[7] != 0 || s[8] != 63) return "unsupported spectral selection";
                // default_decompress_parms, 3 components: JFIF means YCbCr; else Adobe transform 0 means RGB (1 and any other
                // value YCbCr); else component ids 'R' 'G' 'B' mean RGB, any others YCbCr
                if (j->jfif) j->rgb = false;
                else if (j->adobe) j->rgb = j->adobe_transform == 0;
                else j->rgb = j->id[0] == 'R' && j->id[1] == 'G' && j->id[2] == 'B';
                j->scan = p + i + len;
                j->scan_len = n - (i + len);
                const int H = j->hs[0], V = j->vs[0];
                j->mcux = (j->w + 8 * H - 1) / (8 * H);
                j->mcuy = (j->h + 8 * V - 1) / (8 * V);
                for (int c = 0; c < 3; ++c) {
                    j->pw[c] = j->mcux * j->hs[c] * 8;
                    j->ph[c] = j->mcuy * j->vs[c] * 8;
                    j->blocks[c] = (size_t)(j->pw[c] / 8) * (j->ph[c] / 8);
                }
                return nullptr;
            }
            default:
                if (m >= 0xC2 && m <= 0xCF && m != 0xC8 && m != 0xCC) return "unsupported JPEG process (progressive / lossless / arithmetic)";
                break;   // APPn, COM, ...
        }
        i += len;
    }
    return "truncated JPEG stream";
}

// Entropy-coded segment reader: FF00 -> FF; any other marker stops the feed (zero fill, as libjpeg does).
struct BitReader {
    const uint8_t *p;
    size_t n, i = 0;
    uint64_t acc = 0;
    int cnt = 0;
    bool marker = false;
    BitReader(const uint8_t *p_, size_t n_) : p(p_), n(n_) {}
    inline void fill() {
        while (cnt <= 56) {
            unsigned byte = 0;
            if (!marker && i < n) {
                byte = p[i];
                if (byte == 0xFF) {
                    if (i + 1 < n && p[i + 1] == 0x00) i += 2;
                    else { marker = true; byte = 0; }
                } else {
                    ++i;
                }
            }
            acc |= (uint64_t)byte << (56 - cnt);
            cnt += 8;
        }
    }
    inline unsigned peek(int nb) const { return (unsigned)(acc >> (64 - nb)); }
    inline void drop(int nb) { acc <<= nb; cnt -= nb; }
    inline int receive_extend(int s) {   // F.2.2.1 RECEIVE + EXTEND
        if (cnt < s) fill();
        const int v = (int)peek(s);
        drop(s);
        return v < (1 << (s - 1)) ? v - (1 << s) + 1 : v;
    }
    inline int decode(const HuffTable &t) {   // F.2.2.3 DECODE with a 10-bit lookahead table
        if (cnt < 16) fill();
        const unsigned e = t.look[peek(HUFF_LOOKAHEAD)];
        if (e) {
            drop(e >> 8);
            return e & 0xFF;
        }
        int l = HUFF_LOOKAHEAD + 1;
        int code = (int)peek(l);
        while (l <= 16 && code > t.maxcode[l]) {
            ++l;
            code = (int)peek(l);
        }
        if (l > 16) { drop(16); return 0; }
        drop(l);
        return t.vals[t.valptr[l] + code - t.mincode[l]];
    }
    void restart() {   // byte-align, step over the RSTn marker
        acc = 0;
        cnt = 0;
        if (marker) {
            while (i + 1 < n && !(p[i] == 0xFF && p[i + 1] >= 0xD0 && p[i + 1] <= 0xD7)) ++i;
            i = std::min(n, i + 2);
            marker = false;
        } else if (i + 1 < n && p[i] == 0xFF && p[i + 1] >= 0xD0 && p[i + 1] <= 0xD7) {
            i += 2;
        }
    }
};

// Locates the restart intervals of an entropy-coded segment: iv = {first data byte, end (exclusive)} per interval, as offsets into
// j.scan.  Returns false when the markers do not describe exactly ceil(MCUs / restart) intervals (then the host decodes).
static bool scan_restart_intervals(const JpegHeader &j, std::vector<uint32_t> *iv) {
    iv->clear();
    if (j.restart <= 0 || j.scan_len >= 0xFFFFFFF0ull) return false;
    const size_t want = ((size_t)j.mcux * j.mcuy + j.restart - 1) / j.restart;
    const uint8_t *p = j.scan;
    const size_t n = j.scan_len;
    size_t start = 0, i = 0;
    int expect = 0;
    bool closed = false;
    while (i < n) {
        const uint8_t *ff = static_cast<const uint8_t *>(memchr(p + i, 0xFF, n - i));
        if (!ff) break;
        const size_t at = (size_t)(ff - p);
        size_t k = at + 1;
        while (k < n && p[k] == 0xFF) ++k;            // fill bytes before a marker
        if (k >= n) break;
        const int m = p[k];
        if (m == 0x00 && k == at + 1) { i = k + 1; continue; }    // stuffed data byte
        if (m >= 0xD0 && m <= 0xD7) {
            if (m - 0xD0 != expect) return false;
            expect = (expect + 1) & 7;
            iv->push_back((uint32_t)start);
            iv->push_back((uint32_t)at);
            start = k + 1;
            i = k + 1;
            continue;
        }
        iv->push_back((uint32_t)start);               // EOI (or any other marker) ends the scan
        iv->push_back((uint32_t)at);
        closed = true;
        break;
    }
    if (!closed) {
        iv->push_back((uint32_t)start);
        iv->push_back((uint32_t)n);
    }
    return iv->size() / 2 == want;
}

static void fill_huff_dev(const JpegHeader &j, JpegHuffDev *d) {
    memset(d, 0, sizeof(*d));
    for (int t = 0; t < 4; ++t) {
        const HuffTable &h = t < 2 ? j.dc[t] : j.ac[t - 2];
        if (!h.present) continue;
        memcpy(d->look[t], h.look, sizeof(h.look));
        memcpy(d->maxleft[t], h.maxleft, sizeof(h.maxleft));
        memcpy(d->mincode[t], h.mincode, sizeof(h.mincode));
        memcpy(d->valptr[t], h.valptr, sizeof(h.valptr));
        memcpy(d->vals[t], h.vals, sizeof(h.vals));
    }
}

// coef: blocks in SCAN order (MCU by MCU: the H*V luma blocks, Cb, Cr), each block 64 int16 in natural order
static void huffman_decode(const JpegHeader &j, int16_t *coef) {
    BitReader b(j.scan, j.scan_len);
    int pred[3] = {0, 0, 0};
    int count = 0;
    for (int my = 0; my < j.mcuy; ++my)
        for (int mx = 0; mx < j.mcux; ++mx) {
            if (j.restart && count && count % j.restart == 0) {
                b.restart();
                pred[0] = pred[1] = pred[2] = 0;
            }
            ++count;
            for (int c = 0; c < 3; ++c) {
                const HuffTable &dct = j.dc[j.td[c]], &act = j.ac[j.ta[c]];
                for (int v = 0; v < j.vs[c]; ++v)
                    for (int hh = 0; hh < j.hs[c]; ++hh) {
                        int16_t *blk = coef;
                        coef += 64;
                        int s = b.decode(dct);
                        if (s) pred[c] += b.receive_extend(s);
                        blk[0] = (int16_t)pred[c];
                        for (int k = 1; k < 64;) {
                            const int rs = b.decode(act);
                            const int r = rs >> 4;
                            s = rs & 15;
                            if (s == 0) {
                                if (r != 15) break;
                                k += 16;
                                continue;
                            }
                            k += r;
                            if (k > 63) break;
                            blk[JZIGZAG[k]] = (int16_t)b.receive_extend(s);
                            ++k;
                        }
                    }
            }
        }
}

// ---- device side --------------------------------------------------------------------------------------------------------
struct JpegImageDev {
    int16_t *coef;             // this image's coefficient blocks (component-major)
    // entropy decoding on the device (streams with restart markers); gpu_entropy == 0: the host filled `coef`
    int gpu_entropy, n_intervals, restart, mcux, mcuy;
    int td[3], ta[3];
    const uint8_t *stream;     // entropy-coded segment (gpu_entropy 1: as received; 2: with the stuffed zero bytes removed, device-made)
    const uint32_t *iv;        // [n_intervals][2]: first byte / end (exclusive) of each restart interval's data, offsets into stream
    int scan_rst;              // gpu_entropy 1: the device locates the markers (jpeg_unstuff_count / scan + jpeg_iv_write_kernel fill iv
    uint32_t *iv_dev;          //   and *n_iv; n_intervals is then the EXPECTED count = the table's capacity)
    const JpegHuffDev *huff;
    // gpu_entropy == 2: self-synchronising decode of a stream WITHOUT restart markers (sub-sequences of SUBSEQ_BITS bits)
    const uint8_t *raw;        // the segment as received (FF 00 stuffing, EOI at the end); raw_len bytes
    uint8_t *clean;            // == stream: jpeg_unstuff_write_kernel fills it
    int raw_len;
    int n_sub;                 // number of sub-sequences            } written on the device by jpeg_unstuff_write_kernel
    long long nbits;           // length of the unstuffed data in bits }
    int *chunk_drop;           // [raw_len / UNSTUFF_CHUNK + 1] non-data bytes per chunk -> (after the scan) before each chunk
    unsigned *exit_state;      // [n_sub] decoder state at the end of each sub-sequence
    unsigned *used_state;      // [n_sub] the start state its last decode began from
    int *sub_blocks;           // [n_sub + 1] blocks completed inside each sub-sequence -> (after the scan) first block of each
    int *changed;              // [0] the last finished round changed some exit state, [1] collects the running round, [2] raw_len - first marker
    // ... of a stream WITH restart markers (rst_sync = its restart interval in MCUs, else 0): the markers are dropped by the
    // unstuff kernels and become known-state boundaries inside the flat chain of sub-sequences
    int rst_sync, iv_cap;
    int *n_iv;                 // [1] restart intervals found (device-written)
    int *iv_start;             // [iv_cap + 2] first CLEAN byte of each interval; [n_iv] = end of the data
    int *chunk_rst;            // [chunks] restart markers per chunk -> (after the scan) before each chunk
    int *seg_dc;               // [3][iv_cap + 1] un-reset DC prefix (mod 2^16) at the last block of each interval, per component
    uint8_t *plane[3];         // component planes, pw x ph
    uint8_t *bgr;              // output frame
    int pw[3], ph[3];
    int nblk[3];               // blocks per component
    int w, h, pitch;           // output geometry
    int H, V;                  // luma sampling factors (chroma is 1x1)
    int rgb;                   // the components are R, G, B: jpeg_color_kernel reorders them instead of converting
    uint16_t qt[3][64];        // per COMPONENT quantisation table, natural order
};

#define JCONST_BITS 13
#define JPASS1_BITS 2
#define JDESCALE(x, n) (((x) + (1 << ((n) - 1))) >> (n))
__device__ __forceinline__ unsigned jpeg_range_limit(int x) {   // sample_range_limit + CENTERJSAMPLE at (x & RANGE_MASK)
    const int m = x & 1023;
    return (unsigned)(m < 128 ? m + 128 : (m < 512 ? 255 : (m < 896 ? 0 : m - 896)));
}
// one 1-D pass of jpeg_idct_islow over 8 values (already dequantised in pass 1); shift = the pass's descale
__device__ __forceinline__ void jpeg_idct_1d(const int *v, int shift, int *o) {
    int z2 = v[2], z3 = v[6];
    int z1 = (z2 + z3) * 4433;
    int tmp2 = z1 + z3 * (-15137), tmp3 = z1 + z2 * 6270;
    int tmp0 = (v[0] + v[4]) << JCONST_BITS, tmp1 = (v[0] - v[4]) << JCONST_BITS;
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    tmp0 = v[7]; tmp1 = v[5]; tmp2 = v[3]; tmp3 = v[1];
    z1 = tmp0 + tmp3;
    z2 = tmp1 + tmp2;
    z3 = tmp0 + tmp2;
    int z4 = tmp1 + tmp3;
    const int z5 = (z3 + z4) * 9633;
    tmp0 *= 2446; tmp1 *= 16819; tmp2 *= 25172; tmp3 *= 12299;
    z1 *= -7373; z2 *= -20995; z3 *= -16069; z4 *= -3196;
    z3 += z5;
    z4 += z5;
    tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
    o[0] = JDESCALE(tmp10 + tmp3, shift); o[7] = JDESCALE(tmp10 - tmp3, shift);
    o[1] = JDESCALE(tmp11 + tmp2, shift); o[6] = JDESCALE(tmp11 - tmp2, shift);
    o[2] = JDESCALE(tmp12 + tmp1, shift); o[5] = JDESCALE(tmp12 - tmp1, shift);
    o[3] = JDESCALE(tmp13 + tmp0, shift); o[4] = JDESCALE(tmp13 - tmp0, shift);
}


__constant__ uint8_t c_zigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                     41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                     30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

__constant__ uint8_t c_unzigzag[64] = {0,  1,  5,  6,  14, 15, 27, 28, 2,  4,  7,  13, 16, 26, 29, 42, 3,  8,  12, 17, 25, 30,
                                       41, 43, 9,  11, 18, 24, 31, 40, 44, 53, 10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38,
                                       46, 51, 55, 60, 21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, 62, 63};

// Coefficient staging of the entropy decoders.  The arena holds the blocks in SCAN order (block n of the scan at coef + 64 n;
// the IDCT and DC kernels map their plane positions to n), each block in natural order.  Every thread assembles its current
// block in a private row of shared memory (33 words apart: the rows of a warp's lanes start in different banks) and the WARP
// writes finished blocks out together: one 128-byte store per block instead of ~30 scattered 2-byte stores, and no per-lane
// pointer bookkeeping in the decode loop.  A block carries its zeros, so nothing pre-clears the arena.
constexpr int STAGE_PITCH = 33;

// all 32 lanes: writes lane `src`'s staged block to `dst` and clears the row.  [kf, ke) != [0, 64): only the coefficients whose
// SCAN position lies in that range (a block shared with the neighbouring sub-sequences, jpeg_write_kernel).
__device__ __forceinline__ void stage_flush(unsigned *stage_warp, int src, int lane, int16_t *dst, int kf, int ke, bool valid) {
    unsigned *w = stage_warp + src * STAGE_PITCH + lane;
    const unsigned word = *w;
    *w = 0u;
    if (!valid) return;
    if (kf == 0 && ke == 64) {
        reinterpret_cast<unsigned *>(dst)[lane] = word;
    } else {
        const int e = 2 * lane, k0 = c_unzigzag[e], k1 = c_unzigzag[e + 1];
        if (k0 >= kf && k0 < ke) dst[e] = (int16_t)(word & 0xFFFFu);
        if (k1 >= kf && k1 < ke) dst[e + 1] = (int16_t)(word >> 16);
    }
}

constexpr int HUFF_THREADS = 64;

// grid (ceil(max intervals / 64), B): one restart interval per thread.
//
// The decode is ONE flat loop that consumes exactly one Huffman symbol per lane per iteration (DC or AC, decided by the lane's
// own position k in its block): the 32 lanes of a warp sit at unrelated points of 32 different bit streams, and a nested
// MCU / block / coefficient loop nest would leave them in different loop levels — i.e. serialised.  In the flat form every lane
// runs the same instructions with predicated updates of k / block / MCU, so the warp stays converged until its lanes run out
// of MCUs.  Codes longer than the lookahead are resolved without a loop (count of the left-aligned length boundaries the
// 16-bit prefix has passed); the refill appends an aligned 32-bit word when none of its bytes is 0xFF (a data FF is followed by
// a stuffed 00 that must be dropped: ~1.6 % of the words) and goes byte by byte otherwise; block pointers advance by
// per-image constants.  What is left to diverge: the FF words, the block advance (~1 iteration in 35 per lane) and the tail.
__global__ void __launch_bounds__(HUFF_THREADS) jpeg_huffman_kernel(const JpegImageDev *__restrict__ imgs) {
    __shared__ JpegHuffDev tab;
    __shared__ unsigned stage[HUFF_THREADS * STAGE_PITCH];
    __shared__ uint8_t zz[64];
    const JpegImageDev &im = imgs[blockIdx.y];
    const int n_intervals = im.scan_rst ? min(im.n_intervals, *im.n_iv) : im.n_intervals;
    if (im.gpu_entropy != 1 || blockIdx.x * HUFF_THREADS >= n_intervals) return;   // uniform over the CTA
    if (threadIdx.x < 64) zz[threadIdx.x] = c_zigzag[threadIdx.x];
    for (int i = threadIdx.x; i < (int)(sizeof(JpegHuffDev) / 4); i += HUFF_THREADS)
        reinterpret_cast<unsigned *>(&tab)[i] = __ldg(reinterpret_cast<const unsigned *>(im.huff) + i);
    for (int i = threadIdx.x; i < HUFF_THREADS * STAGE_PITCH; i += HUFF_THREADS) stage[i] = 0u;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    unsigned *stage_warp = stage + (threadIdx.x & ~31) * STAGE_PITCH;
    int16_t *my_row = reinterpret_cast<int16_t *>(stage + threadIdx.x * STAGE_PITCH);
    const uint16_t *look = &tab.look[0][0];
    const int iv = blockIdx.x * HUFF_THREADS + threadIdx.x;
    const bool live = iv < n_intervals;
    // The interval's bytes are consumed as ALIGNED 32-bit words, each loaded one refill ahead of its use (`wnext`), so the load's
    // latency (DRAM: the stream has just arrived over PCIe) overlaps the ~4 symbols decoded in between.  `lo`/`hi`: the first and
    // one-past-last byte address of the interval; bytes of a word outside [lo, hi) are ignored.
    const uintptr_t lo = reinterpret_cast<uintptr_t>(im.stream) + (live ? im.iv[2 * iv] : 0u);
    const uintptr_t hi = reinterpret_cast<uintptr_t>(im.stream) + (live ? im.iv[2 * iv + 1] : 0u);
    uintptr_t ap = lo & ~(uintptr_t)3;                                  // address of the word in wnext
    unsigned wnext = ap < hi ? *reinterpret_cast<const unsigned *>(ap) : 0u;
    bool ffpending = false;                                            // the previous byte was a data FF: the next one is its stuffed 00
    unsigned long long acc = 0;
    int cnt = 0;
    const int HV = im.H * im.V, per_mcu = HV + 2, restart = im.restart;
    const int ds0 = im.td[0] << HUFF_LOOKAHEAD, ds1 = im.td[1] << HUFF_LOOKAHEAD, ds2 = im.td[2] << HUFF_LOOKAHEAD;
    const int as0 = (2 + im.ta[0]) << HUFF_LOOKAHEAD, as1 = (2 + im.ta[1]) << HUFF_LOOKAHEAD, as2 = (2 + im.ta[2]) << HUFF_LOOKAHEAD;
    int pred0 = 0, pred1 = 0, pred2 = 0;
    const int mcu_end = live ? min((iv + 1) * restart, im.mcux * im.mcuy) : 0;
    int mcu = live ? iv * restart : 0;
    int n = mcu * per_mcu;          // block number in scan order
    int q = 0, k = 0;               // block within the MCU (scan order: HV luma blocks, Cb, Cr), next coefficient (0 = DC)
    bool active = mcu < mcu_end;
    int dslot = ds0, aslot = as0, comp = 0;
    while (__any_sync(0xffffffffu, active)) {
        bool done = false;                                             // this lane finished a block in this iteration
        if (active) {
            // ---- refill: >= 33 valid bits afterwards = one code (<= 16) + one value (<= 15) ----
            while (cnt <= 32) {
                const unsigned w = wnext;
                const uintptr_t wa = ap;
                ap += 4;
                wnext = ap < hi ? *reinterpret_cast<const unsigned *>(ap) : 0u;      // needed one refill from now
                const unsigned inv = ~w;                                               // a byte of w is FF  <=>  that byte of ~w is 00
                if (wa >= lo && wa + 4 <= hi && !ffpending && ((inv - 0x01010101u) & ~inv & 0x80808080u) == 0) {
                    acc |= (unsigned long long)__byte_perm(w, 0, 0x0123) << (32 - cnt);
                    cnt += 32;
                } else if (wa >= hi) {
                    cnt += 32;                                                         // past the interval: zero bits
                } else {                                                               // an FF, or the interval's first / last word
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const unsigned byte = (w >> (8 * i)) & 0xFFu;
                        if (wa + i < lo || wa + i >= hi) continue;
                        if (ffpending) { ffpending = false; continue; }               // the stuffed 00 after a data FF
                        acc |= (unsigned long long)byte << (56 - cnt);
                        cnt += 8;
                        ffpending = byte == 0xFFu;
                    }
                }
            }
            // ---- one symbol ----
            const bool dc = k == 0;
            const int slot = dc ? dslot : aslot;
            const unsigned top16 = (unsigned)(acc >> 48);
            const unsigned e = look[slot + (top16 >> (16 - HUFF_LOOKAHEAD))];
            int len = (int)(e >> 8), sym = (int)(e & 0xFF);
            if (!e) {                                                  // F.2.2.3 DECODE beyond the lookahead, without a loop
                const int t = slot >> HUFF_LOOKAHEAD;
                len = HUFF_LOOKAHEAD + 1;
#pragma unroll
                for (int l = HUFF_LOOKAHEAD + 1; l <= 16; ++l) len += top16 >= tab.maxleft[t][l] ? 1 : 0;
                if (len > 16) { len = 16; sym = 0; }
                else sym = tab.vals[t][tab.valptr[t][len] + (int)(top16 >> (16 - len)) - tab.mincode[t][len]];
            }
            acc <<= len;
            cnt -= len;
            const int s = dc ? sym : (sym & 15), r = dc ? 0 : (sym >> 4);
            int val = 0;
            if (s) {                                                   // F.2.2.1 RECEIVE + EXTEND
                const int v = (int)(acc >> (64 - s));
                acc <<= s;
                cnt -= s;
                val = v < (1 << (s - 1)) ? v - (1 << s) + 1 : v;
            }
            // ---- where it goes ----
            int kk = k + r;                                            // AC: position of this coefficient
            if (dc) {
                const int pred = (comp == 0 ? pred0 : (comp == 1 ? pred1 : pred2)) + val;
                pred0 = comp == 0 ? pred : pred0;
                pred1 = comp == 1 ? pred : pred1;
                pred2 = comp == 2 ? pred : pred2;
                val = pred;
                kk = 0;
            }
            if ((dc || s) && kk < 64) my_row[dc ? 0 : zz[kk]] = (int16_t)val;
            k = dc ? 1 : (s ? kk + 1 : (r == 15 ? k + 16 : 64));       // DC / coefficient / ZRL / EOB
            done = k >= 64;
        }
        unsigned fm = __ballot_sync(0xffffffffu, done);
        if (fm) {
            __syncwarp();
            do {
                const int src = __ffs(fm) - 1;
                fm &= fm - 1;
                int16_t *dst = im.coef + (size_t)__shfl_sync(0xffffffffu, n, src) * 64;
                stage_flush(stage_warp, src, lane, dst, 0, 64, true);
            } while (fm);
            __syncwarp();
        }
        if (done) {                                                    // next block of the scan
            k = 0;
            ++n;
            if (++q == per_mcu) {                                      // next MCU
                q = 0;
                ++mcu;
                active = mcu < mcu_end;
            }
            comp = q < HV ? 0 : q - HV + 1;
            dslot = comp == 0 ? ds0 : (comp == 1 ? ds1 : ds2);
            aslot = comp == 0 ? as0 : (comp == 1 ? as1 : as2);
        }
    }
}


// ---- streams WITHOUT restart markers: self-synchronising parallel Huffman decoding ------------------------------------------
// A Huffman decoder started at an arbitrary bit of the stream, in an arbitrary state, decodes garbage for a while and then
// (with overwhelming probability) falls into step with the true symbol sequence: prefix codes self-synchronise, and so does
// the JPEG state around them (position k in the block, block q in the MCU) because a wrong table breaks the alignment again
// until all three agree.  This is used as follows (Klein & Wiseman's observation, organised for a GPU like Weissenberger &
// Schmidt's decoder):
//   0. the segment crosses PCIe as received; three small kernels remove the byte stuffing (FF 00 -> FF) and find the end of the
//      data (the first marker), so that bit positions are plain offsets and the host never touches the entropy-coded bytes;
//   1. every thread decodes one sub-sequence of SUBSEQ_BITS bits — thread 0 from the true start state, every other thread from
//      a guessed state at its first bit — and records the state in which it crosses the sub-sequence's end;
//   2. rounds: thread i looks at the state thread i-1 recorded; if that is not the state its own last decode started from, it
//      decodes its sub-sequence again from there and records its exit state again.  Thread 0's chain is correct by
//      construction, so after round r the first r+1 exit states are final; in practice almost all of them are final after
//      round 1 and later rounds touch only the few sub-sequences whose input still moves.  The rounds stop when one changes
//      nothing: the states are then THE fixed point of the chain, i.e. exactly what the serial decoder passes through
//      (the fixed point is unique — induction from thread 0 — so reading a neighbour's state while it is being replaced is
//      harmless: either value is a guess, and a changed state always forces another round);
//   3. the same pass counts the blocks finished inside each sub-sequence; an exclusive scan turns the counts into the index of
//      the block each sub-sequence starts in;
//   4. a last pass decodes every sub-sequence from its (now exact) start state and writes the coefficients; DC values are
//      written as differences and integrated per component afterwards (jpeg_dc_kernel).
#ifndef FD_SUBSEQ_BITS
#define FD_SUBSEQ_BITS 4096
#endif
constexpr int SUBSEQ_BITS = FD_SUBSEQ_BITS;   // 2048 / 4096 / 8192 / 16384 measured on the bench's frames: profiles/r2_jpeg_selfsync_subseq.txt

// exclusive prefix sums of a[0..n) in place by one CTA of 1024 threads; returns the total to every thread
__device__ __forceinline__ int block_exclusive_scan_1024(int *a, int n) {
    __shared__ int warp_sums[33];
    __shared__ int carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int base = 0; base < n; base += 1024) {
        const int i = base + threadIdx.x;
        const int v = i < n ? a[i] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int nb = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += nb;
        }
        if (lane == 31) warp_sums[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const int w = warp_sums[lane];
            int wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int nb = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += nb;
            }
            warp_sums[lane] = wi - w;
            if (lane == 31) warp_sums[32] = wi;
        }
        __syncthreads();
        const int carry = carry_s;
        if (i < n) a[i] = carry + warp_sums[warp] + incl - v;
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + warp_sums[32];
        __syncthreads();
    }
    return carry_s;
}

// -- step 0: byte unstuffing on the device.  What jdhuff.c's fill_bit_buffer does with an FF: further FFs are fill bytes, a 00
// after them makes ONE data byte FF, anything else is a marker and ends the data.  Per byte, with its two neighbours:
//   dropped: a 00 that follows an FF (stuffing), an FF that is followed by an FF (fill);  marker: an FF followed by neither.
constexpr int UNSTUFF_THREADS = 256;
constexpr int UNSTUFF_CHUNK = UNSTUFF_THREADS * 16;

// the 16 bytes at [g, g+16) of a raw segment of n bytes (g % 16 == 0, g < n): bit j of *drop / *mark / *rst classifies byte g + j.
// rst_ok (the stream is decoded with its restart markers as boundaries): FF D0..D7 is dropped, both bytes, and flagged in *rst.
__device__ __forceinline__ uint4 unstuff_classify(const uint8_t *__restrict__ raw, int n, int g, bool rst_ok, unsigned *drop, unsigned *mark,
                                                  unsigned *rst) {
    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(raw + g));        // the arena is padded: bytes past n are ignored below
    const unsigned w[4] = {v.x, v.y, v.z, v.w};
    unsigned prev = g > 0 ? __ldg(raw + g - 1) : 0u;
    const unsigned after = g + 16 < n ? __ldg(raw + g + 16) : 1u;
    unsigned d = 0, m = 0, rs = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const unsigned b = (w[j >> 2] >> ((j & 3) * 8)) & 0xFFu;
        unsigned nx = j < 15 ? (w[(j + 1) >> 2] >> (((j + 1) & 3) * 8)) & 0xFFu : after;
        if (g + j + 1 >= n) nx = 1u;                                         // an FF that ends the buffer counts as a marker
        if (g + j < n) {
            const bool rst_here = rst_ok && b == 0xFFu && (nx & 0xF8u) == 0xD0u;
            const bool rst_tail = rst_ok && prev == 0xFFu && (b & 0xF8u) == 0xD0u;
            if ((b == 0u && prev == 0xFFu) || (b == 0xFFu && nx == 0xFFu) || rst_here || rst_tail) d |= 1u << j;
            else if (b == 0xFFu && nx != 0u) m |= 1u << j;
            if (rst_here) rs |= 1u << j;
        }
        prev = b;
    }
    *drop = d;
    *mark = m;
    *rst = rs;
    return v;
}

// grid (chunks covering [0, raw_len], B): non-data bytes per chunk, and the first marker (changed[2] = raw_len - position, 0 = none)
__global__ void __launch_bounds__(UNSTUFF_THREADS) jpeg_unstuff_count_kernel(const JpegImageDev *__restrict__ imgs) {
    const JpegImageDev &im = imgs[blockIdx.y];
    const int n = im.raw_len;
    if (!(im.gpu_entropy == 2 || im.scan_rst) || (long long)blockIdx.x * UNSTUFF_CHUNK > n) return;
    const int g = blockIdx.x * UNSTUFF_CHUNK + threadIdx.x * 16;
    const bool rst_ok = im.rst_sync != 0 || im.scan_rst != 0;
    unsigned drop = 0, mark = 0, rst = 0;
    if (g < n) unstuff_classify(im.raw, n, g, rst_ok, &drop, &mark, &rst);
    int cnt = __popc(drop), nr = __popc(rst);
    int slack = mark ? n - (g + __ffs(mark) - 1) : 0;                        // larger = earlier
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        nr += __shfl_xor_sync(0xffffffffu, nr, o);
        slack = max(slack, __shfl_xor_sync(0xffffffffu, slack, o));
    }
    __shared__ int s_cnt[UNSTUFF_THREADS / 32], s_nr[UNSTUFF_THREADS / 32], s_slack[UNSTUFF_THREADS / 32];
    if ((threadIdx.x & 31) == 0) { s_cnt[threadIdx.x >> 5] = cnt; s_nr[threadIdx.x >> 5] = nr; s_slack[threadIdx.x >> 5] = slack; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < UNSTUFF_THREADS / 32; ++w) { cnt += s_cnt[w]; nr += s_nr[w]; slack = max(slack, s_slack[w]); }
        im.chunk_drop[blockIdx.x] = cnt;
        if (rst_ok) im.chunk_rst[blockIdx.x] = nr;
        if (slack) atomicMax(im.changed + 2, slack);
    }
}

// one CTA per image: chunk counts -> non-data bytes before each chunk
__global__ void __launch_bounds__(1024) jpeg_unstuff_scan_kernel(const JpegImageDev *__restrict__ imgs) {
    const JpegImageDev &im = imgs[blockIdx.x];
    if (!(im.gpu_entropy == 2 || im.scan_rst)) return;
    if (im.gpu_entropy == 2) block_exclusive_scan_1024(im.chunk_drop, im.raw_len / UNSTUFF_CHUNK + 1);
    if (im.rst_sync || im.scan_rst) block_exclusive_scan_1024(im.chunk_rst, im.raw_len / UNSTUFF_CHUNK + 1);
}

// the data bytes before the first marker, compacted; the thread that owns the end position publishes nbits / n_sub and pads
__global__ void __launch_bounds__(UNSTUFF_THREADS) jpeg_unstuff_write_kernel(JpegImageDev *__restrict__ imgs) {
    JpegImageDev &im = imgs[blockIdx.y];
    const int n = im.raw_len;
    if (im.gpu_entropy != 2) return;
    const int end = n - im.changed[2];                                       // first marker (not RSTn when those are boundaries), or raw_len
    if ((long long)blockIdx.x * UNSTUFF_CHUNK > end) return;
    const int g = blockIdx.x * UNSTUFF_CHUNK + threadIdx.x * 16;
    const bool rst_ok = im.rst_sync != 0;
    unsigned drop = 0, mark = 0, rst = 0;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (g < n) v = unstuff_classify(im.raw, n, g, rst_ok, &drop, &mark, &rst);
    const int cnt = __popc(drop), nr = __popc(rst);
    int incl = cnt, incl_r = nr;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int nb = __shfl_up_sync(0xffffffffu, incl, o), nbr = __shfl_up_sync(0xffffffffu, incl_r, o);
        if (lane >= o) { incl += nb; incl_r += nbr; }
    }
    __shared__ int s_w[UNSTUFF_THREADS / 32], s_r[UNSTUFF_THREADS / 32];
    if (lane == 31) { s_w[warp] = incl; s_r[warp] = incl_r; }
    __syncthreads();
    int before = im.chunk_drop[blockIdx.x] + incl - cnt;                     // non-data bytes before byte g
    int rbefore = rst_ok ? im.chunk_rst[blockIdx.x] + incl_r - nr : 0;       // restart markers before byte g
    for (int w = 0; w < warp; ++w) { before += s_w[w]; rbefore += s_r[w]; }
    uint8_t *out = im.clean;
    if (end >= g && end < g + 16) {
        const unsigned below = (1u << (end - g)) - 1u;
        const int ulen = end - before - __popc(drop & below);
        im.nbits = (long long)ulen * 8;
        im.n_sub = (int)(((long long)ulen * 8 + SUBSEQ_BITS - 1) / SUBSEQ_BITS);
        for (int j = 0; j < 32; ++j) out[ulen + j] = 0;                      // the decoders read a few words past the end
        if (rst_ok) {
            const int niv = min(rbefore + __popc(rst & below) + 1, im.iv_cap);
            *im.n_iv = niv;
            im.iv_start[0] = 0;
            im.iv_start[niv] = ulen;
        }
    }
    const unsigned w[4] = {v.x, v.y, v.z, v.w};
    int o = g - before;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        if (g + j < end) {
            if ((rst >> j) & 1u) {                                           // interval rbefore + 1 starts where this marker was
                ++rbefore;
                if (rbefore < im.iv_cap) im.iv_start[rbefore] = o;
            }
            if (!((drop >> j) & 1u)) out[o++] = (uint8_t)(w[j >> 2] >> ((j & 3) * 8));
        }
    }
}

// One-interval-per-thread decoding (gpu_entropy 1, scan_rst): the restart-interval table from the same marker classification,
// as RAW byte offsets {first data byte, end} — interval j+1 starts behind marker j, the last one ends at the first other marker.
__global__ void __launch_bounds__(UNSTUFF_THREADS) jpeg_iv_write_kernel(const JpegImageDev *__restrict__ imgs) {
    const JpegImageDev &im = imgs[blockIdx.y];
    const int n = im.raw_len;
    if (im.gpu_entropy != 1 || !im.scan_rst) return;
    const int end = n - im.changed[2];
    if ((long long)blockIdx.x * UNSTUFF_CHUNK > end) return;
    const int g = blockIdx.x * UNSTUFF_CHUNK + threadIdx.x * 16;
    unsigned drop = 0, mark = 0, rst = 0;
    if (g < n) unstuff_classify(im.raw, n, g, true, &drop, &mark, &rst);
    const int nr = __popc(rst);
    int incl_r = nr;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int nbr = __shfl_up_sync(0xffffffffu, incl_r, o);
        if (lane >= o) incl_r += nbr;
    }
    __shared__ int s_r[UNSTUFF_THREADS / 32];
    if (lane == 31) s_r[warp] = incl_r;
    __syncthreads();
    int rbefore = im.chunk_rst[blockIdx.x] + incl_r - nr;                    // restart markers before byte g
    for (int w = 0; w < warp; ++w) rbefore += s_r[w];
    const int cap = im.n_intervals;
    if (end >= g && end < g + 16) {
        const int niv = min(rbefore + __popc(rst & ((1u << (end - g)) - 1u)) + 1, cap);
        *im.n_iv = niv;
        im.iv_dev[0] = 0u;
        im.iv_dev[2 * niv - 1] = (uint32_t)end;
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        if (g + j < end && ((rst >> j) & 1u)) {
            if (rbefore + 1 < cap) {
                im.iv_dev[2 * rbefore + 1] = (uint32_t)(g + j);              // interval rbefore ends at the marker ...
                im.iv_dev[2 * rbefore + 2] = (uint32_t)(g + j + 2);          // ... and the next one starts behind it
            }
            ++rbefore;
        }
    }
}

constexpr int SYNC_THREADS = 128;
constexpr int RST_SYNC_MIN_MCUS = 32;   // restart intervals from this many MCUs take the self-synchronising decoder (FD_JPEG_RST_SYNC_MIN)

// exit state: bits past the sub-sequence end (< 32) | block-in-MCU q << 5 | coefficient position k << 8
__device__ __forceinline__ unsigned pack_state(int over, int q, int k) { return (unsigned)over | ((unsigned)q << 5) | ((unsigned)k << 8); }

// One Huffman symbol + its value bits from the left-aligned window `acc` (>= 32 valid bits): F.2.2.3 DECODE with the 10-bit
// lookahead (codes beyond it: count of the left-aligned length boundaries the 16-bit prefix has passed) and F.2.2.1 RECEIVE +
// EXTEND.  dc: DC table slot, else AC.  Returns the bits consumed; *s / *r: size and run, *val: the extended value.
__device__ __forceinline__ int huff_symbol(const JpegHuffDev &tab, const uint16_t *look, int slot, bool dc, unsigned long long &acc, int *s_out,
                                           int *r_out, int *val_out) {
    const unsigned top16 = (unsigned)(acc >> 48);
    const unsigned e = look[slot + (top16 >> (16 - HUFF_LOOKAHEAD))];
    int len = (int)(e >> 8), sym = (int)(e & 0xFF);
    if (!e) {
        const int t = slot >> HUFF_LOOKAHEAD;
        len = HUFF_LOOKAHEAD + 1;
#pragma unroll
        for (int l = HUFF_LOOKAHEAD + 1; l <= 16; ++l) len += top16 >= tab.maxleft[t][l] ? 1 : 0;
        if (len > 16) { len = 16; sym = 0; }
        else sym = tab.vals[t][tab.valptr[t][len] + (int)(top16 >> (16 - len)) - tab.mincode[t][len]];
    }
    acc <<= len;
    const int s = dc ? sym : (sym & 15);
    int val = 0;
    if (s) {
        const int v = (int)(acc >> (64 - s));
        acc <<= s;
        val = v < (1 << (s - 1)) ? v - (1 << s) + 1 : v;
    }
    *s_out = s;
    *r_out = dc ? 0 : (sym >> 4);
    *val_out = val;
    return len + s;
}

// Restart intervals as boundaries of the self-synchronising chain (streams decoded with rst_sync): the interval that starts at
// clean byte iv_start[t] begins in a KNOWN decoder state (first block of an MCU, byte-aligned) whatever came before.  A decoder
// takes the boundary when it has overshot it, or when it stands at the end of an MCU with less than a byte to go (the padding
// bits; a whole MCU needs more).  first index t with iv_start[t] * 8 > pos:
__device__ __forceinline__ int rst_next_boundary(const JpegImageDev &im, long long pos) {
    const int n_iv = __ldcg(im.n_iv), byte = (int)(pos >> 3);
    int lo = 1, hi = n_iv + 1;                           // answer in [1, n_iv + 1]
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldcg(im.iv_start + mid) > byte) hi = mid;
        else lo = mid + 1;
    }
    return lo;
}
__device__ __forceinline__ long long rst_boundary_bit(const JpegImageDev &im, int t) {
    return t <= __ldcg(im.n_iv) ? (long long)__ldcg(im.iv_start + t) * 8 : 0x7fffffffffffffffll;
}

// Decodes from bit `pos` in state (q, k) until the position reaches `end_bit`, without storing anything.  Returns the exit
// state; *blocks = blocks finished.
template <bool RST>
__device__ __forceinline__ unsigned decode_subsequence(const JpegImageDev &im, const JpegHuffDev &tab, const uint16_t *look, long long pos,
                                                       long long end_bit, int q, int k, int *blocks) {
    const int HV = im.H * im.V, per_mcu = HV + 2;
    const int ds[3] = {im.td[0] << HUFF_LOOKAHEAD, im.td[1] << HUFF_LOOKAHEAD, im.td[2] << HUFF_LOOKAHEAD};
    const int as[3] = {(2 + im.ta[0]) << HUFF_LOOKAHEAD, (2 + im.ta[1]) << HUFF_LOOKAHEAD, (2 + im.ta[2]) << HUFF_LOOKAHEAD};
    // bit window over the (clean) stream: 64-bit accumulator, left-aligned; aligned big-endian words
    const unsigned *wp = reinterpret_cast<const unsigned *>(im.stream) + (pos >> 5);
    unsigned long long acc = ((unsigned long long)__byte_perm(wp[0], 0, 0x0123) << 32) | __byte_perm(wp[1], 0, 0x0123);
    unsigned wnext = wp[2];                               // loaded one refill ahead of its use (the arena is padded past the end)
    wp += 3;
    int cnt = 64 - (int)(pos & 31);
    acc <<= (int)(pos & 31);
    int comp = q < HV ? 0 : q - HV + 1;
    int dslot = ds[comp], aslot = as[comp];
    int nblocks = 0;
    int t = 0;
    long long bnd = 0x7fffffffffffffffll;
    if (RST) {
        t = rst_next_boundary(im, pos);
        bnd = rst_boundary_bit(im, t);
    }
    while (pos < end_bit) {
        if (RST && (pos >= bnd || ((k | q) == 0 && bnd - pos < 8))) {      // the next interval starts here, in the known state
            pos = bnd;
            q = k = 0;
            dslot = ds[0];
            aslot = as[0];
            wp = reinterpret_cast<const unsigned *>(im.stream) + (pos >> 5);   // (byte-aligned)
            acc = ((unsigned long long)__byte_perm(wp[0], 0, 0x0123) << 32) | __byte_perm(wp[1], 0, 0x0123);
            wnext = wp[2];
            wp += 3;
            cnt = 64 - (int)(pos & 31);
            acc <<= (int)(pos & 31);
            bnd = rst_boundary_bit(im, ++t);
            continue;
        }
        if (cnt <= 32) {
            acc |= (unsigned long long)__byte_perm(wnext, 0, 0x0123) << (32 - cnt);
            cnt += 32;
            wnext = *wp++;
        }
        const bool dc = k == 0;
        int s, r, val;
        const int used = huff_symbol(tab, look, dc ? dslot : aslot, dc, acc, &s, &r, &val);
        cnt -= used;
        pos += used;
        k = dc ? 1 : (s ? k + r + 1 : (r == 15 ? k + 16 : 64));
        if (k >= 64) {
            k = 0;
            ++nblocks;
            if (++q == per_mcu) q = 0;
            comp = q < HV ? 0 : q - HV + 1;
            dslot = ds[comp];
            aslot = as[comp];
        }
    }
    *blocks = nblocks;
    return pack_state((int)(pos - end_bit), q, k);
}

// grid (ceil(max n_sub / 128), B).  round 0: guessed start states (position = first bit, q = k = 0); round > 0: the exit state
// the left neighbour holds now, and only if it differs from the state this sub-sequence was last decoded from.
template <bool RST>
__global__ void __launch_bounds__(SYNC_THREADS) jpeg_sync_kernel(const JpegImageDev *__restrict__ imgs, int round) {
    __shared__ JpegHuffDev tab;
    const JpegImageDev &im = imgs[blockIdx.y];
    if (im.gpu_entropy != 2 || (im.rst_sync != 0) != RST || blockIdx.x * SYNC_THREADS >= im.n_sub) return;
    if (round > 1 && *im.changed == 0) return;          // this image's states are already the fixed point
    const int i = blockIdx.x * SYNC_THREADS + threadIdx.x;
    unsigned st = 0;
    bool work = i < im.n_sub;
    if (work && round > 0) {
        st = i > 0 ? *reinterpret_cast<volatile unsigned *>(im.exit_state + i - 1) : 0u;
        work = st != im.used_state[i];
    }
    if (!__syncthreads_or(work)) return;                 // nothing moved on this CTA's left: skip the table load too
    for (int t = threadIdx.x; t < (int)(sizeof(JpegHuffDev) / 4); t += SYNC_THREADS)
        reinterpret_cast<unsigned *>(&tab)[t] = __ldg(reinterpret_cast<const unsigned *>(im.huff) + t);
    __syncthreads();
    if (!work) return;
    const long long pos = (long long)i * SUBSEQ_BITS + (st & 31u);
    const long long end_bit = min((long long)(i + 1) * SUBSEQ_BITS, im.nbits);
    int blocks = 0;
    const unsigned out = decode_subsequence<RST>(im, tab, &tab.look[0][0], pos, end_bit, (int)((st >> 5) & 7u), (int)(st >> 8), &blocks);
    im.used_state[i] = st;
    if (round == 0 || out != im.exit_state[i]) {
        im.exit_state[i] = out;
        if (round > 0) atomicOr(im.changed + 1, 1);      // [1] collects this round's changes
    }
    im.sub_blocks[i] = blocks;
}

// one CTA per image: publishes the round's change flag ([0] <- [1], [1] <- 0); with do_scan, turns the block counts into
// exclusive prefix sums (sub_blocks[i] = number of the block sub-sequence i starts in)
__global__ void __launch_bounds__(1024) jpeg_sync_epilogue_kernel(const JpegImageDev *__restrict__ imgs, int do_scan) {
    const JpegImageDev &im = imgs[blockIdx.x];
    if (im.gpu_entropy != 2) return;
    if (!do_scan) {
        if (threadIdx.x == 0) { im.changed[0] = im.changed[1]; im.changed[1] = 0; }
        return;
    }
    const int total = block_exclusive_scan_1024(im.sub_blocks, im.n_sub);
    if (threadIdx.x == 0) im.changed[3] = total;          // blocks the stream really holds (the IDCT zeroes the rest)
}

// the write pass: every sub-sequence from its exact start state.  A block that straddles sub-sequences is written piecewise:
// each decoder owns the scan positions [k at its start, k at its end) — zeros included — so the pieces are disjoint and
// together cover the block; whole blocks leave as one 128-byte warp store (stage_flush).
template <bool RST>
__global__ void __launch_bounds__(SYNC_THREADS) jpeg_write_kernel(const JpegImageDev *__restrict__ imgs) {
    __shared__ JpegHuffDev tab;
    __shared__ unsigned stage[SYNC_THREADS * STAGE_PITCH];
    __shared__ uint8_t zz[64];
    const JpegImageDev &im = imgs[blockIdx.y];
    if (im.gpu_entropy != 2 || (im.rst_sync != 0) != RST || blockIdx.x * SYNC_THREADS >= im.n_sub) return;
    if (threadIdx.x < 64) zz[threadIdx.x] = c_zigzag[threadIdx.x];
    for (int t = threadIdx.x; t < (int)(sizeof(JpegHuffDev) / 4); t += SYNC_THREADS)
        reinterpret_cast<unsigned *>(&tab)[t] = __ldg(reinterpret_cast<const unsigned *>(im.huff) + t);
    for (int t = threadIdx.x; t < SYNC_THREADS * STAGE_PITCH; t += SYNC_THREADS) stage[t] = 0u;
    __syncthreads();
    const uint16_t *look = &tab.look[0][0];
    const int lane = threadIdx.x & 31;
    unsigned *stage_warp = stage + (threadIdx.x & ~31) * STAGE_PITCH;
    int16_t *my_row = reinterpret_cast<int16_t *>(stage + threadIdx.x * STAGE_PITCH);
    const int i = blockIdx.x * SYNC_THREADS + threadIdx.x;
    const bool live = i < im.n_sub;
    const int HV = im.H * im.V, per_mcu = HV + 2;
    const int total_blocks = RST ? im.mcux * im.mcuy * per_mcu : min(im.mcux * im.mcuy * per_mcu, im.changed[3]);
    const int ds0 = im.td[0] << HUFF_LOOKAHEAD, ds1 = im.td[1] << HUFF_LOOKAHEAD, ds2 = im.td[2] << HUFF_LOOKAHEAD;
    const int as0 = (2 + im.ta[0]) << HUFF_LOOKAHEAD, as1 = (2 + im.ta[1]) << HUFF_LOOKAHEAD, as2 = (2 + im.ta[2]) << HUFF_LOOKAHEAD;
    long long pos = (long long)i * SUBSEQ_BITS;
    int q = 0, k = 0;
    if (live && i > 0) {
        const unsigned st = im.exit_state[i - 1];
        pos += st & 31u;
        q = (st >> 5) & 7u;
        k = (int)(st >> 8);
    }
    const long long end_bit = live ? min((long long)(i + 1) * SUBSEQ_BITS, im.nbits) : 0;
    int n = live ? im.sub_blocks[i] : 0;                  // number (scan order) of the block the start lies in
    int kfirst = k;                                       // first scan position of the current block this thread owns
    int dslot = q < HV ? ds0 : (q == HV ? ds1 : ds2), aslot = q < HV ? as0 : (q == HV ? as1 : as2);
    const unsigned *wp = reinterpret_cast<const unsigned *>(im.stream) + (live ? (pos >> 5) : 0);
    unsigned long long acc = ((unsigned long long)__byte_perm(wp[0], 0, 0x0123) << 32) | __byte_perm(wp[1], 0, 0x0123);
    unsigned wnext = wp[2];                               // loaded one refill ahead of its use
    wp += 3;
    int cnt = 64 - (int)(pos & 31);
    acc <<= (int)(pos & 31);
    bool active = live && pos < end_bit;
    int t = 0;                                            // RST: next restart boundary (see decode_subsequence)
    long long bnd = 0x7fffffffffffffffll;
    if (RST && live) {
        t = rst_next_boundary(im, pos);
        bnd = rst_boundary_bit(im, t);
    }
    while (__any_sync(0xffffffffu, active)) {
        bool done = false;
        if (RST && active && (pos >= bnd || ((k | q) == 0 && bnd - pos < 8))) {
            // interval t starts here: block t * restart * (blocks per MCU), known state.  (A block left unfinished can only come
            // from a corrupt stream: its staged coefficients are dropped.)
            if (k != 0 || kfirst != 0)
                for (int wi = 0; wi < 32; ++wi) reinterpret_cast<unsigned *>(my_row)[wi] = 0u;
            pos = bnd;
            q = k = 0;
            kfirst = 0;
            n = t * im.rst_sync * per_mcu;
            dslot = ds0;
            aslot = as0;
            wp = reinterpret_cast<const unsigned *>(im.stream) + (pos >> 5);
            acc = ((unsigned long long)__byte_perm(wp[0], 0, 0x0123) << 32) | __byte_perm(wp[1], 0, 0x0123);
            wnext = wp[2];
            wp += 3;
            cnt = 64 - (int)(pos & 31);
            acc <<= (int)(pos & 31);
            bnd = rst_boundary_bit(im, ++t);
            active = pos < end_bit;
        } else if (active) {
            if (cnt <= 32) {
                acc |= (unsigned long long)__byte_perm(wnext, 0, 0x0123) << (32 - cnt);
                cnt += 32;
                wnext = *wp++;
            }
            const bool dc = k == 0;
            int s, r, val;
            const int used = huff_symbol(tab, look, dc ? dslot : aslot, dc, acc, &s, &r, &val);
            cnt -= used;
            pos += used;
            const int kk = dc ? 0 : k + r;
            if ((dc || s) && kk < 64) my_row[dc ? 0 : zz[kk]] = (int16_t)val;   // DC: the difference (jpeg_dc_kernel integrates)
            k = dc ? 1 : (s ? kk + 1 : (r == 15 ? k + 16 : 64));
            done = k >= 64;
            active = pos < end_bit;
        }
        unsigned fm = __ballot_sync(0xffffffffu, done);
        if (fm) {
            __syncwarp();
            do {
                const int src = __ffs(fm) - 1;
                fm &= fm - 1;
                const int ns = __shfl_sync(0xffffffffu, n, src);
                const int kf = __shfl_sync(0xffffffffu, kfirst, src);
                stage_flush(stage_warp, src, lane, im.coef + (size_t)ns * 64, kf, 64, ns < total_blocks);
            } while (fm);
            __syncwarp();
        }
        if (done) {                                                          // next block of the scan
            k = 0;
            kfirst = 0;
            ++n;
            if (++q == per_mcu) q = 0;
            dslot = q < HV ? ds0 : (q == HV ? ds1 : ds2);
            aslot = q < HV ? as0 : (q == HV ? as1 : as2);
        }
    }
    // the block each sub-sequence ends in: positions [kfirst, k) are this thread's, the successor continues at k
    unsigned fm = __ballot_sync(0xffffffffu, live && k > kfirst);
    __syncwarp();
    while (fm) {
        const int src = __ffs(fm) - 1;
        fm &= fm - 1;
        const int ns = __shfl_sync(0xffffffffu, n, src);
        const int kf = __shfl_sync(0xffffffffu, kfirst, src);
        const int ke = __shfl_sync(0xffffffffu, min(k, 64), src);
        stage_flush(stage_warp, src, lane, im.coef + (size_t)ns * 64, kf, ke, ns < total_blocks);
    }
}

// DC prediction (T.81 F.2.1.3.1: DIFF is relative to the previous block OF THE SAME COMPONENT in scan order; no restart markers
// here, so one chain per component over the whole image): grid (3 components, B), the write pass left the differences in blk[0].
__global__ void __launch_bounds__(1024) jpeg_dc_kernel(const JpegImageDev *__restrict__ imgs) {
    const JpegImageDev &im = imgs[blockIdx.y];
    if (im.gpu_entropy != 2) return;
    const int c = blockIdx.x;
    const int HV = im.H * im.V, per_mcu = HV + 2;
    const int per = c == 0 ? HV : 1;                       // blocks of this component per MCU
    const int total = im.mcux * im.mcuy * per;
    __shared__ int warp_sums[33];
    __shared__ int carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int b0 = 0; b0 < total; b0 += 1024) {
        const int n = b0 + threadIdx.x;                    // index in the component's scan order
        int16_t *blk = nullptr;
        int v = 0;
        if (n < total) {
            const int mcu = n / per, sub = n - mcu * per;
            blk = im.coef + ((size_t)mcu * per_mcu + (c == 0 ? sub : HV + c - 1)) * 64;
            v = blk[0];
        }
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int nb = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += nb;
        }
        if (lane == 31) warp_sums[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const int w = warp_sums[lane];
            int wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int nb = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += nb;
            }
            warp_sums[lane] = wi - w;
            if (lane == 31) warp_sums[32] = wi;
        }
        __syncthreads();
        const int carry = carry_s;
        if (blk) {
            const int p = carry + warp_sums[warp] + incl;
            blk[0] = (int16_t)p;
            if (im.rst_sync) {   // restart intervals reset the predictors: the IDCT subtracts the prefix at the previous interval's last block
                const int mcu = n / per, sub = n - mcu * per;
                if (sub == per - 1 && ((mcu + 1) % im.rst_sync == 0 || mcu == im.mcux * im.mcuy - 1))
                    im.seg_dc[c * (im.iv_cap + 1) + mcu / im.rst_sync] = p;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + warp_sums[32];
        __syncthreads();
    }
}

constexpr int IDCT_BLOCKS = 32;   // DCT blocks per CTA (8 threads each)

// grid (ceil(blocks of the image / 32), B): thread = (block, column) in pass 1, (block, row) in pass 2
__global__ void __launch_bounds__(IDCT_BLOCKS * 8) jpeg_idct_kernel(const JpegImageDev *__restrict__ imgs) {
    __shared__ int ws[IDCT_BLOCKS][64 + 8];   // +8: the row pass reads 8 consecutive ints per thread, rows of different blocks apart
    const JpegImageDev &im = imgs[blockIdx.y];
    const int lb = threadIdx.x >> 3, k = threadIdx.x & 7;
    const int gb = blockIdx.x * IDCT_BLOCKS + lb;
    const int total = im.nblk[0] + im.nblk[1] + im.nblk[2];
    const bool live = gb < total;
    // the arena is in scan order (the CTA reads 32 consecutive blocks = 4 KB): block n -> component c, block (yb, xb) of its plane
    const int n = gb, HV = im.H * im.V;
    const int mcu = n / (HV + 2), qb = n - mcu * (HV + 2);
    const int my = mcu / im.mcux, mx = mcu - my * im.mcux;
    const int c = qb < HV ? 0 : qb - HV + 1;
    const int yb = c == 0 ? my * im.V + qb / im.H : my, xb = c == 0 ? mx * im.H + qb % im.H : mx;
    if (live) {
        bool held = im.gpu_entropy != 2 || im.rst_sync != 0 || n < im.changed[3];   // a truncated stream holds fewer blocks: the rest is zero
        if (im.gpu_entropy == 1 && im.scan_rst && mcu / im.restart >= *im.n_iv) held = false;   // ... or fewer restart intervals
        int dc_base = 0;                                      // (rst_sync: the arena was cleared instead)
        if (im.gpu_entropy == 2 && im.rst_sync != 0 && k == 0) {
            const int seg = mcu / im.rst_sync;
            if (seg > 0) dc_base = im.seg_dc[c * (im.iv_cap + 1) + seg - 1];
        }
        const int16_t *in = im.coef + (size_t)n * 64 + k;             // column k of the block
        const uint16_t *q = im.qt[c] + k;
        int v[8], o[8];
        bool ac0 = true;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            int cf = held ? (int)in[8 * r] : 0;
            if (r == 0 && k == 0) cf = (int)(int16_t)(cf - dc_base);   // modular: both are un-reset prefixes mod 2^16
            v[r] = cf * (int)q[8 * r];                        // DEQUANTIZE
            if (r) ac0 = ac0 && cf == 0;
        }
        if (ac0) {   // jidctint.c's shortcut (identical to the general path for an all-zero AC column)
            const int dc = v[0] << JPASS1_BITS;
#pragma unroll
            for (int r = 0; r < 8; ++r) o[r] = dc;
        } else {
            jpeg_idct_1d(v, JCONST_BITS - JPASS1_BITS, o);
        }
#pragma unroll
        for (int r = 0; r < 8; ++r) ws[lb][8 * r + k] = o[r];
    }
    __syncthreads();
    if (!live) return;
    int v[8], o[8];
#pragma unroll
    for (int x = 0; x < 8; ++x) v[x] = ws[lb][8 * k + x];     // row k
    jpeg_idct_1d(v, JCONST_BITS + JPASS1_BITS + 3, o);
    uint8_t *dst = im.plane[c] + (size_t)(yb * 8 + k) * im.pw[c] + xb * 8;
    uint2 out;
    out.x = jpeg_range_limit(o[0]) | (jpeg_range_limit(o[1]) << 8) | (jpeg_range_limit(o[2]) << 16) | (jpeg_range_limit(o[3]) << 24);
    out.y = jpeg_range_limit(o[4]) | (jpeg_range_limit(o[5]) << 8) | (jpeg_range_limit(o[6]) << 16) | (jpeg_range_limit(o[7]) << 24);
    *reinterpret_cast<uint2 *>(dst) = out;                   // planes are 8-byte aligned, pw % 8 == 0
}

// chroma sample at full resolution (jdsample.c fullsize / h2v1_fancy / h2v2_fancy, jdmainct.c context rows)
__device__ __forceinline__ int jpeg_chroma_at(const uint8_t *__restrict__ pl, int pitch, int dw, int dh, int H, int V, int x, int y) {
    if (H == 1) return pl[(size_t)y * pitch + x];
    const int cx = x >> 1;
    if (dw <= 2) return pl[(size_t)(V == 2 ? y >> 1 : y) * pitch + cx];   // jinit_upsampler: replication for narrow components
    if (V == 1) {
        const uint8_t *r = pl + (size_t)y * pitch;
        const int v = r[cx];
        if (!(x & 1)) return cx == 0 ? v : (v * 3 + r[cx - 1] + 1) >> 2;
        if (cx == 0) return (v * 3 + r[1] + 2) >> 2;
        return cx == dw - 1 ? v : (v * 3 + r[cx + 1] + 2) >> 2;
    }
    const int cy = y >> 1;
    int ny = (y & 1) ? cy + 1 : cy - 1;
    ny = max(0, min(dh - 1, ny));
    const uint8_t *r0 = pl + (size_t)cy * pitch, *r1 = pl + (size_t)ny * pitch;
    const int t = r0[cx] * 3 + r1[cx];
    if (cx == 0) return (x & 1) ? (t * 3 + (r0[1] * 3 + r1[1]) + 7) >> 4 : (t * 4 + 8) >> 4;
    if (!(x & 1)) return (t * 3 + (r0[cx - 1] * 3 + r1[cx - 1]) + 8) >> 4;
    return cx == dw - 1 ? (t * 4 + 7) >> 4 : (t * 3 + (r0[cx + 1] * 3 + r1[cx + 1]) + 7) >> 4;
}

__device__ __forceinline__ unsigned jpeg_ycc_to_bgr(int Y, int cb, int cr) {   // jdcolor.c: cb, cr already minus 128
    const int r = Y + ((91881 * cr + 32768) >> 16);                        // FIX(1.40200)
    const int g = Y + ((-22554 * cb + 32768 + -46802 * cr) >> 16);         // -FIX(0.34414), -FIX(0.71414)
    const int b = Y + ((116130 * cb + 32768) >> 16);                       // FIX(1.77200)
    return (unsigned)max(0, min(255, b)) | ((unsigned)max(0, min(255, g)) << 8) | ((unsigned)max(0, min(255, r)) << 16);
}

// The six column sums 3*near + far (h2v2_fancy_upsample's thiscolsum) of chroma columns cx0-1 .. cx0+4, from one aligned word
// per row plus the two edge bytes.  cx0 % 4 == 0.
__device__ __forceinline__ void jpeg_colsums6(const uint8_t *__restrict__ r0, const uint8_t *__restrict__ r1, int cx0, int pw, int *cs) {
    const unsigned w0 = *reinterpret_cast<const unsigned *>(r0 + cx0), w1 = *reinterpret_cast<const unsigned *>(r1 + cx0);
    const int lft = max(cx0 - 1, 0), rgt = min(cx0 + 4, pw - 1);
    cs[0] = 3 * r0[lft] + r1[lft];
#pragma unroll
    for (int i = 0; i < 4; ++i) cs[1 + i] = 3 * (int)((w0 >> (8 * i)) & 0xFF) + (int)((w1 >> (8 * i)) & 0xFF);
    cs[5] = 3 * r0[rgt] + r1[rgt];
}

// one output pixel, BGR in the low 24 bits, from the luma / first component and the upsampled other two minus 128.  RGB:
// jdcolor.c rgb_rgb_convert, the components are R, G, B and only change places.
template <bool RGB>
__device__ __forceinline__ unsigned jpeg_to_bgr(int Y, int cb, int cr) {
    if (RGB) return (unsigned)(cr + 128) | ((unsigned)(cb + 128) << 8) | ((unsigned)Y << 16);
    return jpeg_ycc_to_bgr(Y, cb, cr);
}

// grid (ceil(w/8 / 128), h rows, B): 8 pixels per thread -> 24 bytes = six aligned 32-bit stores (pitch % 16 == 0).
// 4:2:0 with downsampled_width > 2 (the common case) shares the triangle filter's column sums between the 8 pixels and reads
// the planes by words; the other samplings take the per-pixel form (jpeg_chroma_at).  One build per colour space: each skips
// the images of the other (the flag is per image, so the exit is uniform over the CTA) and is launched only for batches that
// hold such an image.
template <bool RGB>
__global__ void __launch_bounds__(128) jpeg_color_kernel(const JpegImageDev *__restrict__ imgs) {
    const JpegImageDev &im = imgs[blockIdx.z];
    const int y = blockIdx.y;
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
    if (y >= im.h || x0 >= im.w || (im.rgb != 0) != RGB) return;
    const int H = im.H, V = im.V;
    const int dw = (im.w + H - 1) / H, dh = (im.h + V - 1) / V;
    unsigned px[8];
    const uint8_t *yrow = im.plane[0] + (size_t)y * im.pw[0];
    if (H == 2 && V == 2 && dw > 2) {
        const uint2 yy = *reinterpret_cast<const uint2 *>(yrow + x0);      // x0 % 8 == 0, pw % 8 == 0, plane 64-byte aligned
        const int cy = y >> 1;
        const int ny = max(0, min(dh - 1, (y & 1) ? cy + 1 : cy - 1));
        const int cx0 = x0 >> 1, pw = im.pw[1];
        int cb[6], cr[6];
        jpeg_colsums6(im.plane[1] + (size_t)cy * pw, im.plane[1] + (size_t)ny * pw, cx0, pw, cb);
        jpeg_colsums6(im.plane[2] + (size_t)cy * pw, im.plane[2] + (size_t)ny * pw, cx0, pw, cr);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int cx = cx0 + (j >> 1), t = (j >> 1) + 1, o = (j & 1) ? t + 1 : t - 1;
            const int rnd = (j & 1) ? 7 : 8;
            const bool edge = (j & 1) ? cx == dw - 1 : cx == 0;             // h2v2_fancy_upsample's first / last column cases
            const int vb = edge ? (cb[t] * 4 + rnd) >> 4 : (cb[t] * 3 + cb[o] + rnd) >> 4;
            const int vr = edge ? (cr[t] * 4 + rnd) >> 4 : (cr[t] * 3 + cr[o] + rnd) >> 4;
            const int Y = (int)(((j < 4 ? yy.x : yy.y) >> (8 * (j & 3))) & 0xFF);
            px[j] = jpeg_to_bgr<RGB>(Y, vb - 128, vr - 128);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int x = min(x0 + j, im.w - 1);
            const int cb = jpeg_chroma_at(im.plane[1], im.pw[1], dw, dh, H, V, x, y) - 128;
            const int cr = jpeg_chroma_at(im.plane[2], im.pw[2], dw, dh, H, V, x, y) - 128;
            px[j] = jpeg_to_bgr<RGB>(yrow[x], cb, cr);
        }
    }
    uint8_t *row = im.bgr + (size_t)y * im.pitch;
    if (x0 + 7 < im.w) {
        unsigned *o = reinterpret_cast<unsigned *>(row + (size_t)x0 * 3);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const unsigned *p4 = px + 4 * q;
            o[3 * q + 0] = p4[0] | (p4[1] << 24);
            o[3 * q + 1] = (p4[1] >> 8) | (p4[2] << 16);
            o[3 * q + 2] = (p4[2] >> 16) | (p4[3] << 8);
        }
    } else {
        for (int j = 0; j < 8 && x0 + j < im.w; ++j) {
            row[(x0 + j) * 3] = (uint8_t)px[j];
            row[(x0 + j) * 3 + 1] = (uint8_t)(px[j] >> 8);
            row[(x0 + j) * 3 + 2] = (uint8_t)(px[j] >> 16);
        }
    }
}


// grid (x, B): clears the coefficient blocks of the images decoded with their restart markers as boundaries (a missing interval
// would leave a hole of stale coefficients): 128-bit streaming stores
__global__ void __launch_bounds__(256) jpeg_zero_rst_kernel(const JpegImageDev *__restrict__ imgs) {
    const JpegImageDev &im = imgs[blockIdx.y];
    if (im.gpu_entropy != 2 || im.rst_sync == 0) return;
    const size_t n16 = ((size_t)im.nblk[0] + im.nblk[1] + im.nblk[2]) * 8;       // a block is 128 bytes
    uint4 *p = reinterpret_cast<uint4 *>(im.coef);
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) __stcs(p + i, z);
}

}  // namespace fd

using namespace fd;

FD_EXPORT int fd_jpeg_info(const uint8_t *jpeg, size_t nbytes, int *height, int *width, int *subsampling) {
    FD_REQUIRE(jpeg && height && width, "fd_jpeg_info: null argument");
    JpegHeader *j = new JpegHeader();
    const char *err = parse_jpeg(jpeg, nbytes, j);
    if (!err) {
        *height = j->h;
        *width = j->w;
        if (subsampling) *subsampling = j->hs[0] * 10 + j->vs[0];
    }
    delete j;
    if (err) return fail(FD_ERR_INVALID, std::string("fd_jpeg_info: ") + err);
    return FD_OK;
}

FD_EXPORT int fd_decode_jpeg_batch(fd_ctx *ctx, const uint8_t *const *jpegs, const size_t *nbytes, int B, int n_threads, fd_frame *frames_out) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(jpegs && nbytes && frames_out && B > 0, "fd_decode_jpeg_batch: bad arguments");
    static const bool dbg = getenv("FD_JPEG_DBG") != nullptr;   // host-phase timeline on stderr
    auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_begin = now();
    double t_parse = 0, t_wait = 0, t_copies = 0;
    const int hw_threads = std::max(1, n_threads > 0 ? n_threads : (int)std::thread::hardware_concurrency());
    // runs fn(i) for i in [0, B) on up to hw_threads threads of the calling process (images are independent)
    auto parallel_images = [&](int limit, const std::function<void(int)> &fn) {
        std::atomic<int> next(0);
        auto work = [&]() {
            for (int i = next.fetch_add(1); i < B; i = next.fetch_add(1)) fn(i);
        };
        const int nt = std::max(1, std::min(limit, hw_threads));
        std::vector<std::thread> pool;
        for (int t = 1; t < nt; ++t) pool.emplace_back(work);
        work();
        for (auto &t : pool) t.join();
    };
    static const bool no_gpu_entropy = getenv("FD_JPEG_HOST_HUFFMAN") != nullptr;   // A/B switch: force the host Huffman pass
    static const bool no_selfsync = getenv("FD_JPEG_NO_SELFSYNC") != nullptr;        // A/B switch: host pass for streams without RSTn
    // 0. headers, Huffman tables and (streams with restart markers) the restart-interval table: host parsing, one image per thread.
    //    Entropy-decoding mode per image: 1 = device, one restart interval per thread; 2 = device, self-synchronising sub-sequences
    //    (no restart markers); 0 = host (more than two DC / AC tables, or a restart-marker sequence that does not add up).
    std::vector<JpegHeader> hdr((size_t)B);
    std::vector<const char *> errs((size_t)B, nullptr);
    std::vector<std::vector<uint32_t>> ivs((size_t)B);
    std::vector<char> mode((size_t)B, 0);
    std::vector<int> rst_iv((size_t)B, 0);          // mode 2 on a stream WITH restart markers: its restart interval (MCUs)
    static const int rst_sync_min = getenv("FD_JPEG_RST_SYNC_MIN") ? atoi(getenv("FD_JPEG_RST_SYNC_MIN")) : RST_SYNC_MIN_MCUS;
    static const bool host_marker_scan = getenv("FD_JPEG_HOST_MARKER_SCAN") != nullptr;   // A/B switch: round-2 behaviour (memchr scan, host fallback)
    parallel_images(B, [&](int i) {
        errs[i] = parse_jpeg(jpegs[i], nbytes[i], &hdr[i]);
        if (errs[i]) return;
        const JpegHeader &j = hdr[i];
        bool ok = !no_gpu_entropy && j.scan_len < 0x7FFFFFF0ull;
        for (int c = 0; c < 3 && ok; ++c) ok = j.td[c] <= 1 && j.ta[c] <= 1;
        // long restart intervals (few threads for one-interval-per-thread decoding: 13.9 ms per 64 frames at one MCU row) take the
        // self-synchronising decoder with the markers as boundaries; the device finds the markers, no host scan
        if (ok && j.restart >= rst_sync_min && !no_selfsync) { mode[i] = 2; rst_iv[i] = j.restart; }
        else if (ok && j.restart > 0) mode[i] = host_marker_scan ? (scan_restart_intervals(j, &ivs[i]) ? 1 : 0) : 1;
        else if (ok && !no_selfsync) mode[i] = 2;
    });
    for (int i = 0; i < B; ++i)
        if (errs[i]) return fail(FD_ERR_INVALID, "fd_decode_jpeg_batch: image " + std::to_string(i) + ": " + errs[i]);
    t_parse = now();
    // layout: coefficient arena (device; pinned mirror for host-decoded images), plane arena, frame arena, stream / aux arenas
    std::vector<size_t> coef_off(B), plane_off(B), frame_off(B), stream_off(B), aux_off(B), raw_off(B), sync_off(B);
    size_t coef_total = 0, plane_total = 0, frame_total = 0, stream_total = 0, aux_total = 0, host_coef_total = 0, raw_total = 0, sync_total = 0;
    int max_blocks = 0, max_h = 0, max_w = 0, max_iv = 0, max_sub = 0, max_chunks = 0, n_rst = 0, n_sync = 0, n_rstsync = 0, n_scan = 0, n_rgb = 0;
    for (int i = 0; i < B; ++i) {
        const JpegHeader &j = hdr[i];
        const size_t nblk = j.blocks[0] + j.blocks[1] + j.blocks[2];
        coef_off[i] = coef_total;
        coef_total += nblk * 64;                                   // int16 elements
        plane_off[i] = plane_total;
        plane_total += (nblk * 64 + 255) & ~(size_t)255;           // u8 elements (a plane byte per coefficient)
        frame_off[i] = frame_total;
        const size_t pitch = ((size_t)j.w * 3 + 15) & ~(size_t)15;
        frame_total += (pitch * j.h + 255) & ~(size_t)255;
        max_blocks = std::max<int>(max_blocks, (int)nblk);
        max_h = std::max(max_h, j.h);
        max_w = std::max(max_w, j.w);
        n_rgb += j.rgb ? 1 : 0;
        if (mode[i] == 1) {
            ++n_rst;
            stream_off[i] = stream_total;
            stream_total += (j.scan_len + 15) & ~(size_t)15;
            aux_off[i] = aux_total;
            aux_total += ((sizeof(JpegHuffDev) + ivs[i].size() * sizeof(uint32_t)) + 15) & ~(size_t)15;
            const size_t want = ((size_t)j.mcux * j.mcuy + j.restart - 1) / j.restart;
            max_iv = std::max<int>(max_iv, host_marker_scan ? (int)(ivs[i].size() / 2) : (int)want);
            if (!host_marker_scan) {                   // device marker scan: markers per chunk, flags' neighbours, the interval table
                const size_t nchunks = j.scan_len / UNSTUFF_CHUNK + 1;
                sync_off[i] = sync_total;
                sync_total += (2 * nchunks + 4 + 2 * want + 4) * sizeof(int);
                max_chunks = std::max<int>(max_chunks, (int)nchunks);
                ++n_scan;
            }
        } else if (mode[i] == 2) {
            ++n_sync;
            stream_off[i] = stream_total;
            stream_total += (j.scan_len + 64 + 15) & ~(size_t)15;
            raw_off[i] = raw_total;
            raw_total += (j.scan_len + 32 + 15) & ~(size_t)15;
            aux_off[i] = aux_total;
            aux_total += (sizeof(JpegHuffDev) + 15) & ~(size_t)15;
            const size_t nsub_cap = (j.scan_len * 8 + SUBSEQ_BITS - 1) / SUBSEQ_BITS + 1;
            const size_t nchunks = j.scan_len / UNSTUFF_CHUNK + 1;
            sync_off[i] = sync_total;
            const size_t iv_cap = rst_iv[i] ? ((size_t)j.mcux * j.mcuy + rst_iv[i] - 1) / rst_iv[i] : 0;
            // exit states, start states, block counts; chunk counts; (restart boundaries) interval starts, markers per chunk, DC segment ends
            sync_total += (nsub_cap * 3 + nchunks + 4 + (rst_iv[i] ? (iv_cap + 2) + nchunks + 3 * (iv_cap + 1) + 4 : 0)) * sizeof(int);
            n_rstsync += rst_iv[i] ? 1 : 0;
            max_sub = std::max<int>(max_sub, (int)nsub_cap - 1);
            max_chunks = std::max<int>(max_chunks, (int)nchunks);
        } else {
            host_coef_total += nblk * 64;
        }
    }
    const int n_gpu = n_rst + n_sync;
    FD_TRY(ctx->jpeg_coef_host.reserve(std::max<size_t>(host_coef_total, 1) * sizeof(int16_t)));
    FD_TRY(ctx->jpeg_coef.reserve(coef_total * sizeof(int16_t)));
    FD_TRY(ctx->jpeg_planes.reserve(plane_total));
    FD_TRY(ctx->jpeg_frames.reserve(frame_total + 256));
    FD_TRY(ctx->jpeg_desc.reserve(sizeof(JpegImageDev) * (size_t)B));
    FD_TRY(ctx->jpeg_desc_host.reserve(sizeof(JpegImageDev) * (size_t)B));
    FD_TRY(ctx->jpeg_stream.reserve(stream_total + 64));
    FD_TRY(ctx->jpeg_aux.reserve(aux_total + 64));
    FD_TRY(ctx->jpeg_aux_host.reserve(aux_total + 64));
    FD_TRY(ctx->jpeg_raw.reserve(raw_total + 64));
    FD_TRY(ctx->jpeg_sync.reserve(sync_total + 64));
    FD_TRY(ctx->jpeg_flags.reserve(sizeof(int) * 4 * (size_t)B));
    FD_TRY(ctx->jpeg_flags_host.reserve(sizeof(int) * 4 * (size_t)B));
    const double t_layout = now();
    FD_CUDA(cudaEventSynchronize(ctx->ev[3]));   // the previous call's H2D copies have left the pinned staging buffers
    t_wait = now();
    int64_t h2d = 0;
    // 1a. device paths: the entropy-coded segments go up as they are
    if (n_gpu) {
        unsigned char *aux = ctx->jpeg_aux_host.as<unsigned char>();
        // (one copy queue: alternating the copies over two streams was measured 2x SLOWER, 5.0 vs 2.4 ms for 64 x 1.26 MB)
        for (int i = 0; i < B; ++i) {
            if (!mode[i]) continue;
            fill_huff_dev(hdr[i], reinterpret_cast<JpegHuffDev *>(aux + aux_off[i]));
            if (mode[i] == 1) memcpy(aux + aux_off[i] + sizeof(JpegHuffDev), ivs[i].data(), ivs[i].size() * sizeof(uint32_t));
            uint8_t *dst = mode[i] == 1 ? ctx->jpeg_stream.as<uint8_t>() + stream_off[i] : ctx->jpeg_raw.as<uint8_t>() + raw_off[i];
            if (hdr[i].scan_len) FD_CUDA(cudaMemcpyAsync(dst, hdr[i].scan, hdr[i].scan_len, cudaMemcpyHostToDevice, ctx->stream));
            h2d += (int64_t)hdr[i].scan_len;
        }
        FD_CUDA(cudaMemcpyAsync(ctx->jpeg_aux.p, aux, aux_total, cudaMemcpyHostToDevice, ctx->stream));
        h2d += (int64_t)aux_total;
        if (n_sync || n_scan) FD_CUDA(cudaMemsetAsync(ctx->jpeg_flags.p, 0, sizeof(int) * 4 * (size_t)B, ctx->stream));
    }
    // 1b. host path: entropy decoding on the host, images are independent, one per worker thread
    std::vector<size_t> host_off(B, 0);
    if (n_gpu < B) {
        int16_t *coef_host = ctx->jpeg_coef_host.as<int16_t>();
        size_t o = 0;
        for (int i = 0; i < B; ++i)
            if (!mode[i]) { host_off[i] = o; o += (hdr[i].blocks[0] + hdr[i].blocks[1] + hdr[i].blocks[2]) * 64; }
        parallel_images(B - n_gpu, [&](int i) {
            if (mode[i]) return;
            const size_t n = (hdr[i].blocks[0] + hdr[i].blocks[1] + hdr[i].blocks[2]) * 64;
            memset(coef_host + host_off[i], 0, n * sizeof(int16_t));
            huffman_decode(hdr[i], coef_host + host_off[i]);
        });
        for (int i = 0; i < B; ++i) {
            if (mode[i]) continue;
            const size_t n = (hdr[i].blocks[0] + hdr[i].blocks[1] + hdr[i].blocks[2]) * 64;
            FD_CUDA(cudaMemcpyAsync(ctx->jpeg_coef.as<int16_t>() + coef_off[i], coef_host + host_off[i], n * sizeof(int16_t), cudaMemcpyHostToDevice,
                                    ctx->stream));
            h2d += (int64_t)(n * sizeof(int16_t));
        }
    }
    if (ctx->trace_on) trace_mark(ctx, __FILE__, __LINE__, "jpeg_h2d_copies");
    t_copies = now();
    // 2. descriptors
    JpegImageDev *desc = ctx->jpeg_desc_host.as<JpegImageDev>();
    for (int i = 0; i < B; ++i) {
        const JpegHeader &j = hdr[i];
        JpegImageDev &d = desc[i];
        memset(&d, 0, sizeof(d));
        d.coef = ctx->jpeg_coef.as<int16_t>() + coef_off[i];
        uint8_t *pl = ctx->jpeg_planes.as<uint8_t>() + plane_off[i];
        for (int c = 0; c < 3; ++c) {
            d.plane[c] = pl;
            pl += j.blocks[c] * 64;
            d.pw[c] = j.pw[c];
            d.ph[c] = j.ph[c];
            d.nblk[c] = (int)j.blocks[c];
            d.td[c] = j.td[c];
            d.ta[c] = j.ta[c];
            memcpy(d.qt[c], j.qt[j.tq[c]], sizeof(d.qt[c]));
        }
        d.w = j.w;
        d.h = j.h;
        d.pitch = (j.w * 3 + 15) & ~15;
        d.bgr = ctx->jpeg_frames.as<uint8_t>() + frame_off[i];
        d.H = j.hs[0];
        d.V = j.vs[0];
        d.rgb = j.rgb ? 1 : 0;
        d.mcux = j.mcux;
        d.mcuy = j.mcuy;
        d.restart = j.restart;
        d.gpu_entropy = mode[i];
        if (mode[i]) {
            d.stream = ctx->jpeg_stream.as<uint8_t>() + stream_off[i];
            d.huff = reinterpret_cast<const JpegHuffDev *>(ctx->jpeg_aux.as<unsigned char>() + aux_off[i]);
        }
        if (mode[i] == 1 && host_marker_scan) {
            d.n_intervals = (int)(ivs[i].size() / 2);
            d.iv = reinterpret_cast<const uint32_t *>(ctx->jpeg_aux.as<unsigned char>() + aux_off[i] + sizeof(JpegHuffDev));
        } else if (mode[i] == 1) {
            const size_t nchunks = j.scan_len / UNSTUFF_CHUNK + 1;
            int *p = reinterpret_cast<int *>(ctx->jpeg_sync.as<unsigned char>() + sync_off[i]);
            d.scan_rst = 1;
            d.raw = d.stream;
            d.raw_len = (int)j.scan_len;
            d.n_intervals = (int)(((size_t)j.mcux * j.mcuy + j.restart - 1) / j.restart);
            d.chunk_drop = p;
            d.chunk_rst = p + nchunks;
            d.n_iv = d.chunk_rst + nchunks;
            d.iv_dev = reinterpret_cast<uint32_t *>(d.n_iv + 4);
            d.iv = d.iv_dev;
            d.changed = ctx->jpeg_flags.as<int>() + 4 * i;
        } else if (mode[i] == 2) {
            d.raw = ctx->jpeg_raw.as<uint8_t>() + raw_off[i];
            d.clean = ctx->jpeg_stream.as<uint8_t>() + stream_off[i];
            d.raw_len = (int)j.scan_len;
            d.nbits = 0;                                            // both set by jpeg_unstuff_write_kernel
            d.n_sub = 0;
            const size_t cap = (j.scan_len * 8 + SUBSEQ_BITS - 1) / SUBSEQ_BITS + 1;
            unsigned *sy = reinterpret_cast<unsigned *>(ctx->jpeg_sync.as<unsigned char>() + sync_off[i]);
            d.exit_state = sy;
            d.used_state = sy + cap;
            d.sub_blocks = reinterpret_cast<int *>(sy + 2 * cap);
            d.chunk_drop = reinterpret_cast<int *>(sy + 3 * cap);
            if (rst_iv[i]) {
                const size_t nchunks = j.scan_len / UNSTUFF_CHUNK + 1;
                d.rst_sync = rst_iv[i];
                d.iv_cap = (int)(((size_t)j.mcux * j.mcuy + rst_iv[i] - 1) / rst_iv[i]);
                int *p = d.chunk_drop + nchunks;
                d.n_iv = p;
                d.iv_start = p + 4;
                d.chunk_rst = d.iv_start + d.iv_cap + 2;
                d.seg_dc = d.chunk_rst + nchunks;
            }
            d.changed = ctx->jpeg_flags.as<int>() + 4 * i;
        }
        frames_out[i].data = d.bgr;
        frames_out[i].height = j.h;
        frames_out[i].width = j.w;
        frames_out[i].pitch = d.pitch;
    }
    FD_CUDA(cudaMemcpyAsync(ctx->jpeg_desc.p, desc, sizeof(JpegImageDev) * (size_t)B, cudaMemcpyHostToDevice, ctx->stream));
    FD_CUDA(cudaEventRecord(ctx->ev[3], ctx->stream));
    h2d += (int64_t)(sizeof(JpegImageDev) * (size_t)B);
    ctx->jpeg_last_h2d = h2d;
    ctx->jpeg_last_gpu_entropy = n_gpu;
    ctx->jpeg_last_selfsync = n_sync;
    ctx->jpeg_last_B = B;
    const JpegImageDev *ddesc = ctx->jpeg_desc.as<JpegImageDev>();
    // 3a. entropy decoding on the device, streams with (short) restart intervals: the device locates the markers, then one
    //     restart interval per thread
    if (n_sync || n_scan) {
        dim3 gu(max_chunks, B);
        jpeg_unstuff_count_kernel<<<gu, UNSTUFF_THREADS, 0, ctx->stream>>>(ddesc);
        FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_unstuff_count_kernel");
        jpeg_unstuff_scan_kernel<<<B, 1024, 0, ctx->stream>>>(ddesc);
        FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_unstuff_scan_kernel");
        if (n_scan) {
            jpeg_iv_write_kernel<<<gu, UNSTUFF_THREADS, 0, ctx->stream>>>(ddesc);
            FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_iv_write_kernel");
        }
    }
    if (n_rst) {
        dim3 g0((max_iv + HUFF_THREADS - 1) / HUFF_THREADS, B);
        jpeg_huffman_kernel<<<g0, HUFF_THREADS, 0, ctx->stream>>>(ddesc);
        FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_huffman_kernel");
    }
    // 3b. streams without restart markers: unstuff on the device, then self-synchronising rounds until one changes no exit state
    //     (rounds are enqueued in groups — a round with nothing to do costs a few microseconds — and the flags read once per
    //     group), then count -> scan -> write -> DC prefix
    ctx->jpeg_last_rounds = 0;
    if (n_sync) {
        dim3 gu(max_chunks, B);
        jpeg_unstuff_write_kernel<<<gu, UNSTUFF_THREADS, 0, ctx->stream>>>(ctx->jpeg_desc.as<JpegImageDev>());
        FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_unstuff_write_kernel");
    }
    if (n_sync && max_sub > 0) {
        dim3 gs((max_sub + SYNC_THREADS - 1) / SYNC_THREADS, B);
        const bool plain = n_sync > n_rstsync, rsts = n_rstsync > 0;       // which builds of the decoders this batch needs
        auto sync_round = [&](int r) -> int {
            if (plain) jpeg_sync_kernel<false><<<gs, SYNC_THREADS, 0, ctx->stream>>>(ddesc, r);
            if (rsts) jpeg_sync_kernel<true><<<gs, SYNC_THREADS, 0, ctx->stream>>>(ddesc, r);
            FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_sync_kernel");
            return FD_OK;
        };
        if (rsts) {
            jpeg_zero_rst_kernel<<<dim3(32, B), 256, 0, ctx->stream>>>(ddesc);
            FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_zero_rst_kernel");
        }
        FD_TRY(sync_round(0));
        int round = 0;
        int *flags = ctx->jpeg_flags_host.as<int>();
        for (int group = 6;; group = 4) {
            for (int r = 0; r < group; ++r) {
                ++round;
                FD_TRY(sync_round(round));
                jpeg_sync_epilogue_kernel<<<B, 32, 0, ctx->stream>>>(ddesc, 0);
                FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_sync_epilogue_kernel");
            }
            FD_CUDA(cudaMemcpyAsync(flags, ctx->jpeg_flags.p, sizeof(int) * 4 * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
            FD_CUDA(cudaStreamSynchronize(ctx->stream));
            bool any = false;
            for (int i = 0; i < B; ++i) any = any || (mode[i] == 2 && flags[4 * i] != 0);
            if (!any) break;
            FD_REQUIRE(round <= max_sub + 8, "fd_decode_jpeg_batch: the sub-sequence states did not converge (corrupt stream?)");
        }
        ctx->jpeg_last_rounds = round;
        jpeg_sync_epilogue_kernel<<<B, 1024, 0, ctx->stream>>>(ddesc, 1);
        FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_sync_epilogue_kernel");
        if (plain) jpeg_write_kernel<false><<<gs, SYNC_THREADS, 0, ctx->stream>>>(ddesc);
        if (rsts) jpeg_write_kernel<true><<<gs, SYNC_THREADS, 0, ctx->stream>>>(ddesc);
        FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_write_kernel");
        jpeg_dc_kernel<<<dim3(3, B), 1024, 0, ctx->stream>>>(ddesc);
        FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_dc_kernel");
    }
    // 4. IDCT, upsampling + colour conversion
    dim3 g1((max_blocks + IDCT_BLOCKS - 1) / IDCT_BLOCKS, B);
    jpeg_idct_kernel<<<g1, IDCT_BLOCKS * 8, 0, ctx->stream>>>(ddesc);
    FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_idct_kernel");
    FD_REQUIRE(max_h <= 65535 && B <= 65535, "fd_decode_jpeg_batch: image too tall / batch too large for one launch");
    dim3 g2(((max_w + 7) / 8 + 127) / 128, max_h, B);
    if (n_rgb < B) {
        jpeg_color_kernel<false><<<g2, 128, 0, ctx->stream>>>(ddesc);
        FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_color_kernel");
    }
    if (n_rgb) {
        jpeg_color_kernel<true><<<g2, 128, 0, ctx->stream>>>(ddesc);
        FD_LAUNCH_CHECK_NAMED(ctx, "jpeg_color_kernel");
    }
    if (dbg)
        fprintf(stderr, "[jpeg dbg] B=%d on-device entropy %d: parse+scan %.2f ms, layout %.2f, wait prev copies %.2f, enqueue copies (+host huffman) %.2f, "
                        "descriptors+launches %.2f, total host %.2f ms\n", B, n_gpu, t_parse - t_begin, t_layout - t_parse, t_wait - t_layout,
                t_copies - t_wait, now() - t_copies, now() - t_begin);
    return FD_OK;
}

FD_EXPORT int fd_jpeg_last_stats(const fd_ctx *ctx, int64_t *out) {
    FD_REQUIRE(ctx && out, "fd_jpeg_last_stats: null");
    out[0] = ctx->jpeg_last_h2d;
    out[1] = ctx->jpeg_last_gpu_entropy;
    out[2] = ctx->jpeg_last_B - ctx->jpeg_last_gpu_entropy;
    out[3] = ((int64_t)ctx->jpeg_last_rounds << 32) | (unsigned)ctx->jpeg_last_selfsync;
    return FD_OK;
}

FD_EXPORT int fd_imdecode(fd_ctx *ctx, const uint8_t *jpeg, size_t nbytes, uint8_t *out_bgr, int pitch) {
    FD_TRY(check_ctx(ctx));
    FD_REQUIRE(jpeg && out_bgr, "fd_imdecode: null argument");
    fd_frame fr;
    FD_TRY(fd_decode_jpeg_batch(ctx, &jpeg, &nbytes, 1, 1, &fr));
    FD_REQUIRE(pitch >= fr.width * 3, "fd_imdecode: pitch smaller than a row");
    FD_CUDA(cudaMemcpy2DAsync(out_bgr, (size_t)pitch, fr.data, (size_t)fr.pitch, (size_t)fr.width * 3, (size_t)fr.height, cudaMemcpyDeviceToHost,
                              ctx->stream));
    FD_CUDA(cudaStreamSynchronize(ctx->stream));
    return FD_OK;
}
