// yf_jpeg.cuh — baseline JPEG decoding on the device, byte-identical to cv2.imdecode(buf, IMREAD_COLOR) (libjpeg-turbo with OpenCV's
// settings: JDCT_ISLOW, fancy upsampling, BGR output). DESIGN.md §5.7.
//
//   host    jpeg_parse: the headers of one file -> JpegDesc (geometry, sampling, restart interval, offsets of the scan data and of the
//           quantisation and Huffman tables inside the file), or a reason why the file is not taken. Nothing is enqueued for a batch
//           until every header has passed.
//   kernel  jpeg_entropy_kernel: one thread decodes one file's scan from start to end (Huffman tables built from the file's DHT bytes,
//           or the ITU-T T.81 K.3 tables when the file has none, RSTn handled in-stream) into quantised coefficients, 128 bytes per
//           8x8 block, in natural order (jdhuff.c).
//   kernel  jpeg_idct_kernel: one thread per block: dequantisation + jpeg_idct_islow (jidctint.c), the 64 samples written in place over
//           the first half of the block's coefficients.
//   kernel  jpeg_color_kernel: one thread per output pixel: h2v1 / h2v2 fancy upsampling of the chroma (jdsample.c) and the fixed-point
//           YCbCr -> RGB tables (jdcolor.c), written B, G, R; gray files write Y three times.
//
// The per-block arithmetic is __host__ __device__ so that it can be checked against cv2 on a machine without a GPU; the library itself
// only ever runs it on the device.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <cstring>
#include <string>

namespace yf {

constexpr int JPEG_CHUNK = 256;                         // descriptors per launch: 256 x 88 bytes of __grid_constant__ parameters
constexpr int JPEG_MAX_SIDE = 16384;                    // the limit of prep_frames_kernel
constexpr int JPEG_STATUS_CORRUPT = 4;                  // YF_STATUS_JPEG_CORRUPT

// Huffman table reference of a component: >= 0 offset in the file of the table's 16 count bytes (the symbols follow); < 0 one of the
// standard tables, -1 - k with k = 0 DC luminance, 1 AC luminance, 2 DC chrominance, 3 AC chrominance (jstdhuff.c)
struct JpegDesc {
    int64_t src;                // offset of the file in the staged bytes
    int64_t dst;                // offset of the BGR frame in the output buffer
    int64_t cbase;              // first block of the file in the coefficient workspace (relative to the launch's chunk)
    int32_t scan, scan_end;     // entropy-coded data [scan, scan_end) within the file
    uint16_t h, w;
    uint16_t mcux, mcuy;        // MCUs per row / column (gray: blocks)
    uint16_t ri;                // restart interval in MCUs (0: none)
    uint8_t ncomp, hs, vs;      // 1 or 3 components; luma sampling factors (chroma 1x1)
    uint8_t qprec;              // bit c: component c's quantisation table has 16-bit entries
    int32_t q[3];               // offset in the file of each component's 64 quantisation values (zigzag order)
    int32_t dc[3], ac[3];       // Huffman tables of each component
};
static_assert(sizeof(JpegDesc) == 88, "JpegDesc layout");
struct JpegChunk { JpegDesc d[JPEG_CHUNK]; };

// standard tables (T.81 K.3; libjpeg jstdhuff.c): 16 counts then the symbols, DC luma, AC luma, DC chroma, AC chroma
#define YF_JPEG_STD_TABLES                                                                                                             \
    {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0,  \
     1, 125, 1, 2, 3, 0, 4, 17, 5, 18, 33, 49, 65, 6, 19, 81, 97, 7, 34, 113, 20, 50, 129, 145, 161, 8, 35, 66, 177, 193, 21, 82,    \
     209, 240, 36, 51, 98, 114, 130, 9, 10, 22, 23, 24, 25, 26, 37, 38, 39, 40, 41, 42, 52, 53, 54, 55, 56, 57, 58, 67, 68, 69, 70,  \
     71, 72, 73, 74, 83, 84, 85, 86, 87, 88, 89, 90, 99, 100, 101, 102, 103, 104, 105, 106, 115, 116, 117, 118, 119, 120, 121, 122,  \
     131, 132, 133, 134, 135, 136, 137, 138, 146, 147, 148, 149, 150, 151, 152, 153, 154, 162, 163, 164, 165, 166, 167, 168, 169,    \
     170, 178, 179, 180, 181, 182, 183, 184, 185, 186, 194, 195, 196, 197, 198, 199, 200, 201, 202, 210, 211, 212, 213, 214, 215,    \
     216, 217, 218, 225, 226, 227, 228, 229, 230, 231, 232, 233, 234, 241, 242, 243, 244, 245, 246, 247, 248, 249, 250, 0, 3, 1, 1,  \
     1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 119, 0,  \
     1, 2, 3, 17, 4, 5, 33, 49, 6, 18, 65, 81, 7, 97, 113, 19, 34, 50, 129, 8, 20, 66, 145, 161, 177, 193, 9, 35, 51, 82, 240, 21,   \
     98, 114, 209, 10, 22, 36, 52, 225, 37, 241, 23, 24, 25, 26, 38, 39, 40, 41, 42, 53, 54, 55, 56, 57, 58, 67, 68, 69, 70, 71, 72,  \
     73, 74, 83, 84, 85, 86, 87, 88, 89, 90, 99, 100, 101, 102, 103, 104, 105, 106, 115, 116, 117, 118, 119, 120, 121, 122, 130,     \
     131, 132, 133, 134, 135, 136, 137, 138, 146, 147, 148, 149, 150, 151, 152, 153, 154, 162, 163, 164, 165, 166, 167, 168, 169,    \
     170, 178, 179, 180, 181, 182, 183, 184, 185, 186, 194, 195, 196, 197, 198, 199, 200, 201, 202, 210, 211, 212, 213, 214, 215,    \
     216, 217, 218, 226, 227, 228, 229, 230, 231, 232, 233, 234, 242, 243, 244, 245, 246, 247, 248, 249, 250}
// natural order of the zigzag index, with 16 extra entries so that a run past coefficient 63 lands on 63 (jutils.c)
#define YF_JPEG_NATURAL                                                                                                                \
    {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,  7,  14, 21, 28,  \
     35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63,  \
     63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63}
static const uint8_t h_jpeg_std[412] = YF_JPEG_STD_TABLES;
static const uint8_t h_jpeg_natural[80] = YF_JPEG_NATURAL;
__constant__ uint8_t c_jpeg_std[412] = YF_JPEG_STD_TABLES;
__constant__ uint8_t c_jpeg_natural[80] = YF_JPEG_NATURAL;

__host__ __device__ inline const uint8_t* jpeg_std_tables() {
#ifdef __CUDA_ARCH__
    return c_jpeg_std;
#else
    return h_jpeg_std;
#endif
}
__host__ __device__ inline int jpeg_natural(int k) {
#ifdef __CUDA_ARCH__
    return c_jpeg_natural[k];
#else
    return h_jpeg_natural[k];
#endif
}

// ---------------------------------------------------------------------------------------------------------------------------------
// host: header parser
// ---------------------------------------------------------------------------------------------------------------------------------
inline int jpeg_rd16(const uint8_t* p) { return (p[0] << 8) | p[1]; }

// EXIF orientation of an APP1 "Exif\0\0" payload: 1..8, 1 when the tag is absent, -1 when the TIFF structure cannot be read
inline int jpeg_exif_orientation(const uint8_t* t, int64_t n) {
    if (n < 8) return -1;
    const bool le = t[0] == 'I' && t[1] == 'I';
    if (!le && !(t[0] == 'M' && t[1] == 'M')) return -1;
    auto u16 = [&](int64_t o) { return le ? (t[o] | (t[o + 1] << 8)) : ((t[o] << 8) | t[o + 1]); };
    auto u32 = [&](int64_t o) {
        return le ? ((uint32_t)t[o] | ((uint32_t)t[o + 1] << 8) | ((uint32_t)t[o + 2] << 16) | ((uint32_t)t[o + 3] << 24))
                  : (((uint32_t)t[o] << 24) | ((uint32_t)t[o + 1] << 16) | ((uint32_t)t[o + 2] << 8) | (uint32_t)t[o + 3]);
    };
    if (u16(2) != 42) return -1;
    const int64_t ifd = u32(4);
    if (ifd < 8 || ifd + 2 > n) return -1;
    const int cnt = u16(ifd);
    if (ifd + 2 + 12 * (int64_t)cnt > n) return -1;
    for (int i = 0; i < cnt; ++i) {
        const int64_t e = ifd + 2 + 12 * (int64_t)i;
        if (u16(e) == 0x0112) return u16(e + 8);         // SHORT, count 1: the value sits in the first bytes of the value field
    }
    return 1;
}

// Parses the headers of one file. Returns true and fills d (all but src / dst / cbase), or false with the reason in `why`.
inline bool jpeg_parse(const uint8_t* f, int64_t n, JpegDesc& d, std::string& why) {
    auto fail = [&](const char* fmt, int a = 0, int b = 0, int c = 0) {
        char buf[256];
        snprintf(buf, sizeof buf, fmt, a, b, c);
        why = buf;
        return false;
    };
    if (!f || n < 4 || f[0] != 0xFF || f[1] != 0xD8) return fail("not a JPEG file (no SOI marker)");
    if (n > 0x7FFFFFFF) return fail("file larger than 2 GB");
    memset(&d, 0, sizeof d);
    int32_t qoff[4] = {-1, -1, -1, -1};
    int qprec[4] = {0, 0, 0, 0};
    int32_t hoff[2][4] = {{-1, -1, -1, -1}, {-1, -1, -1, -1}};
    bool jfif = false, adobe = false, sof = false;
    int adobe_t = -1, ncomp = 0, ri = 0, H = 0, W = 0;
    int cid[3] = {0, 0, 0}, hsf[3] = {0, 0, 0}, vsf[3] = {0, 0, 0}, tq[3] = {0, 0, 0};
    int64_t pos = 2;
    for (;;) {
        if (pos >= n) return fail("truncated header: the file ends before its SOS marker");
        if (f[pos] != 0xFF) return fail("malformed header: stray bytes between markers");
        while (pos < n && f[pos] == 0xFF) ++pos;        // fill bytes
        if (pos >= n) return fail("truncated header: the file ends inside a marker");
        const int m = f[pos++];
        if (m == 0xD9) return fail("malformed header: EOI before SOS");
        if (m == 0x00 || m == 0x01 || m == 0xD8 || (m >= 0xD0 && m <= 0xD7)) return fail("malformed header: unexpected marker 0xFF%02X", m);
        if (pos + 2 > n) return fail("truncated header: the file ends inside a segment length");
        const int L = jpeg_rd16(f + pos);
        if (L < 2 || pos + L > n) return fail("truncated header: segment 0xFF%02X of %d bytes runs past the end of the file", m, L);
        const uint8_t* s = f + pos + 2;
        const int sl = L - 2;
        const int32_t so = (int32_t)(pos + 2);
        if (m == 0xCC || (m >= 0xC9 && m <= 0xCB) || (m >= 0xCD && m <= 0xCF)) return fail("arithmetic-coded JPEG (SOF 0xFF%02X) is not supported", m);
        if (m >= 0xC5 && m <= 0xC7) return fail("hierarchical JPEG (SOF 0xFF%02X) is not supported", m);
        if (m == 0xDE || m == 0xDF) return fail("hierarchical JPEG (marker 0xFF%02X) is not supported", m);
        if (m == 0xC2) return fail("progressive JPEG is not supported");
        if (m == 0xC3) return fail("lossless JPEG is not supported");
        if (m == 0xDC) return fail("DNL marker (height defined after the scan) is not supported");
        if (m == 0xC0 || m == 0xC1) {
            if (sof) return fail("malformed header: two SOF markers");
            if (sl < 6) return fail("malformed SOF segment");
            if (s[0] != 8) return fail("%d-bit samples are not supported (12-bit and other precisions)", s[0]);
            H = jpeg_rd16(s + 1); W = jpeg_rd16(s + 3); ncomp = s[5];
            if (sl != 6 + 3 * ncomp) return fail("malformed SOF segment");
            if (ncomp == 2) return fail("2-component JPEG is not supported");
            if (ncomp == 4) return fail("4-component JPEG (CMYK / YCCK) is not supported");
            if (ncomp != 1 && ncomp != 3) return fail("%d-component JPEG is not supported", ncomp);
            if (H == 0) return fail("height 0 (defined by a DNL marker) is not supported");
            if (W == 0 || H > JPEG_MAX_SIDE || W > JPEG_MAX_SIDE) return fail("size %dx%d outside [1, %d]", H, W, JPEG_MAX_SIDE);
            for (int c = 0; c < ncomp; ++c) {
                cid[c] = s[6 + 3 * c]; hsf[c] = s[7 + 3 * c] >> 4; vsf[c] = s[7 + 3 * c] & 15; tq[c] = s[8 + 3 * c];
                if (hsf[c] < 1 || hsf[c] > 4 || vsf[c] < 1 || vsf[c] > 4 || tq[c] > 3) return fail("malformed SOF segment (component %d)", c);
            }
            if (ncomp == 1 && (hsf[0] != 1 || vsf[0] != 1)) return fail("gray sampling factors %dx%d are not supported", hsf[0], vsf[0]);
            if (ncomp == 3) {
                const bool luma = (hsf[0] == 1 && vsf[0] == 1) || (hsf[0] == 2 && vsf[0] == 1) || (hsf[0] == 2 && vsf[0] == 2);
                if (!luma || hsf[1] != 1 || vsf[1] != 1 || hsf[2] != 1 || vsf[2] != 1) {
                    char buf[160];
                    snprintf(buf, sizeof buf, "sampling factors %dx%d, %dx%d, %dx%d are not supported (4:4:4, 4:2:2 and 4:2:0 are)", hsf[0], vsf[0],
                             hsf[1], vsf[1], hsf[2], vsf[2]);
                    why = buf;
                    return false;
                }
            }
            sof = true;
        } else if (m == 0xC4) {                          // DHT
            int k = 0;
            while (k < sl) {
                const int tc = s[k] >> 4, th = s[k] & 15;
                if (tc > 1 || th > 3 || k + 17 > sl) return fail("malformed DHT segment");
                int total = 0;
                for (int l = 0; l < 16; ++l) total += s[k + 1 + l];
                if (total > 256 || k + 17 + total > sl) return fail("malformed DHT segment");
                int64_t code = 0;                        // jpeg_make_d_derived_tbl: no code may reach all ones of its length
                int last = 0;
                for (int l = 0; l < 16; ++l) if (s[k + 1 + l]) last = l + 1;
                for (int l = 1; l <= last; ++l) {
                    code += s[k + l];
                    if (code >= ((int64_t)1 << l)) return fail("bad Huffman table");
                    code <<= 1;
                }
                if (tc == 0)
                    for (int i = 0; i < total; ++i) if (s[k + 17 + i] > 15) return fail("bad Huffman table (DC symbol above 15)");
                hoff[tc][th] = so + k + 1;
                k += 17 + total;
            }
        } else if (m == 0xDB) {                          // DQT
            int k = 0;
            while (k < sl) {
                const int pq = s[k] >> 4, t = s[k] & 15;
                if (pq > 1 || t > 3 || k + 1 + 64 * (pq + 1) > sl) return fail("malformed DQT segment");
                qoff[t] = so + k + 1; qprec[t] = pq;
                k += 1 + 64 * (pq + 1);
            }
        } else if (m == 0xDD) {                          // DRI
            if (sl != 2) return fail("malformed DRI segment");
            ri = jpeg_rd16(s);
        } else if (m == 0xE0) {
            if (sl >= 14 && memcmp(s, "JFIF\0", 5) == 0) jfif = true;
        } else if (m == 0xEE) {
            if (sl >= 12 && memcmp(s, "Adobe", 5) == 0) { adobe = true; adobe_t = s[11]; }
        } else if (m == 0xE1) {
            if (sl >= 6 && memcmp(s, "Exif\0\0", 6) == 0) {
                const int o = jpeg_exif_orientation(s + 6, sl - 6);
                if (o < 0) return fail("EXIF segment that cannot be read (its orientation is unknown)");
                if (o != 1) return fail("EXIF orientation %d is not supported (cv2 rotates such images)", o);
            }
        } else if (m == 0xDA) {                          // SOS: the header ends here
            if (!sof) return fail("malformed header: SOS before SOF");
            if (sl < 1) return fail("malformed SOS segment");
            const int ns = s[0];
            if (sl != 4 + 2 * ns) return fail("malformed SOS segment");
            if (ns != ncomp) return fail("more than one scan (this scan codes %d of %d components)", ns, ncomp);
            for (int c = 0; c < ns; ++c) {
                if (s[1 + 2 * c] != cid[c]) return fail("malformed SOS segment: components out of frame order");
                const int td = s[2 + 2 * c] >> 4, ta = s[2 + 2 * c] & 15;
                if (td > 3 || ta > 3) return fail("malformed SOS segment");
                if (hoff[0][td] >= 0) d.dc[c] = hoff[0][td];
                else if (td < 2) d.dc[c] = -1 - (td == 0 ? 0 : 2);
                else return fail("undefined DC Huffman table %d", td);
                if (hoff[1][ta] >= 0) d.ac[c] = hoff[1][ta];
                else if (ta < 2) d.ac[c] = -1 - (ta == 0 ? 1 : 3);
                else return fail("undefined AC Huffman table %d", ta);
                if (qoff[tq[c]] < 0) return fail("undefined quantisation table %d", tq[c]);
                d.q[c] = qoff[tq[c]];
                if (qprec[tq[c]]) d.qprec |= (uint8_t)(1 << c);
            }
            const uint8_t* t = s + 1 + 2 * ns;
            if (t[0] != 0 || t[1] != 63 || t[2] != 0) return fail("SOS spectral selection %d..%d / approximation %d is not sequential", t[0], t[1], t[2]);
            pos += L;
            break;
        }
        pos += L;
    }
    if (ncomp == 3) {
        if (adobe && adobe_t == 0) return fail("RGB JPEG (Adobe marker with transform 0) is not supported");
        if (!jfif && !adobe && cid[0] == 'R' && cid[1] == 'G' && cid[2] == 'B') return fail("RGB JPEG (component IDs 'R', 'G', 'B') is not supported");
    }
    // end of the entropy-coded data: the first marker that is not a stuffed 0xFF00 or an RSTn
    const int64_t scan = pos;
    int64_t q = pos;
    while (q < n) {
        const void* ff = memchr(f + q, 0xFF, (size_t)(n - q));
        if (!ff) { q = n; break; }
        q = (const uint8_t*)ff - f;
        if (q + 1 >= n) { q = n; break; }
        const int c = f[q + 1];
        if (c == 0x00 || (c >= 0xD0 && c <= 0xD7)) q += 2;
        else if (c == 0xFF) q += 1;
        else break;
    }
    const int64_t scan_end = q;
    // what follows the scan: EOI, the end of the file, or segments that are not a second scan
    while (q < n) {
        if (f[q] != 0xFF) return fail("malformed data after the scan");
        while (q < n && f[q] == 0xFF) ++q;
        if (q >= n) break;
        const int m = f[q++];
        if (m == 0xD9) break;
        if (m == 0xDA) return fail("more than one scan");
        if (m == 0xDC) return fail("DNL marker (height defined after the scan) is not supported");
        if ((m >= 0xD0 && m <= 0xD8) || m == 0x01 || q + 2 > n) return fail("malformed data after the scan");
        q += jpeg_rd16(f + q);
    }
    d.scan = (int32_t)scan; d.scan_end = (int32_t)scan_end;
    d.h = (uint16_t)H; d.w = (uint16_t)W; d.ri = (uint16_t)ri; d.ncomp = (uint8_t)ncomp;
    d.hs = (uint8_t)hsf[0]; d.vs = (uint8_t)vsf[0];
    d.mcux = (uint16_t)((W + 8 * d.hs - 1) / (8 * d.hs));
    d.mcuy = (uint16_t)((H + 8 * d.vs - 1) / (8 * d.vs));
    return true;
}

// blocks of a file in the coefficient workspace: luma plane (mcux*hs x mcuy*vs blocks), then one plane per chroma component
__host__ __device__ inline int64_t jpeg_blocks(const JpegDesc& d) {
    const int64_t mcus = (int64_t)d.mcux * d.mcuy;
    return d.ncomp == 1 ? mcus : mcus * (d.hs * d.vs + 2);
}

// ---------------------------------------------------------------------------------------------------------------------------------
// stage 1: entropy decoding (jdhuff.c)
// ---------------------------------------------------------------------------------------------------------------------------------
struct JpegHuff {
    uint16_t look[256];         // first 8 bits -> (length << 8) | symbol, 0 for longer codes (HUFF_LOOKAHEAD)
    int32_t maxcode[18];        // largest code of each length, -1 if none; [17] sentinel
    int32_t valoff[17];         // symbol index = code + valoff[length]
    uint8_t val[256];
};

__host__ __device__ inline void jpeg_build_huff(const uint8_t* t, JpegHuff& h) {
    for (int i = 0; i < 256; ++i) h.look[i] = 0;
    int p = 0, code = 0;
    for (int l = 1; l <= 16; ++l) {
        const int cnt = t[l - 1];
        h.valoff[l] = p - code;
        for (int i = 0; i < cnt; ++i, ++p, ++code) {
            const uint8_t sym = t[16 + p];
            h.val[p] = sym;
            if (l <= 8)
                for (int j = code << (8 - l), e = (code + 1) << (8 - l); j < e; ++j) h.look[j] = (uint16_t)((l << 8) | sym);
        }
        h.maxcode[l] = cnt ? code - 1 : -1;
        code <<= 1;
    }
    h.maxcode[17] = 0x7FFFFFFF;
}

// MSB-first bit reader over [pos, end) with libjpeg's marker rules: 0xFF 0x00 is a data 0xFF, further 0xFF fill is skipped, any other
// marker (or the end of the data) stops the reader, which then supplies zero bits. Consuming a supplied zero bit marks the file corrupt.
struct JpegBits {
    const uint8_t* p;
    int64_t pos, end;
    uint64_t buf;
    int nbits, pad;
    bool marker;
    __host__ __device__ inline void fill() {
        while (nbits <= 56) {
            uint32_t c = 0;
            if (!marker) {
                if (pos < end) {
                    c = p[pos];
                    if (c == 0xFF) {
                        int64_t q = pos + 1;
                        while (q < end && p[q] == 0xFF) ++q;
                        if (q < end && p[q] == 0) pos = q + 1;
                        else { marker = true; c = 0; }  // pos stays on the marker's first 0xFF
                    } else {
                        ++pos;
                    }
                } else {
                    marker = true;
                }
            }
            if (marker) pad += 8;
            buf |= (uint64_t)c << (56 - nbits);
            nbits += 8;
        }
    }
    __host__ __device__ inline uint32_t peek(int k) const { return (uint32_t)(buf >> (64 - k)); }
    __host__ __device__ inline void skip(int k) { buf <<= k; nbits -= k; }
    __host__ __device__ inline bool overrun() const { return nbits < pad; }
};

__host__ __device__ inline int jpeg_decode_sym(JpegBits& br, const JpegHuff& h, bool& bad) {
    const uint32_t e = h.look[br.peek(8)];
    if (e) { br.skip(e >> 8); return e & 255; }
    int l = 9;
    int32_t code = (int32_t)br.peek(9);
    while (code > h.maxcode[l]) {
        if (++l > 16) { bad = true; return 0; }
        code = (int32_t)br.peek(l);
    }
    br.skip(l);
    return h.val[code + h.valoff[l]];
}

__host__ __device__ inline int jpeg_extend(int x, int s) { return x < (1 << (s - 1)) ? x + (int)((~0u) << s) + 1 : x; }

__host__ __device__ inline const uint8_t* jpeg_table_bytes(const uint8_t* file, int32_t ref) {
    const int k = -1 - ref;                              // tables of 28, 178, 28 and 178 bytes
    return ref >= 0 ? file + ref : jpeg_std_tables() + (k == 0 ? 0 : k == 1 ? 28 : k == 2 ? 206 : 234);
}

// Decodes one file's scan into `coef` (jpeg_blocks(d) blocks of 64 int16, natural order, quantised as libjpeg stores them). The file
// is read only inside [scan, scan_end). `tabs` holds 2 * ncomp tables of scratch. Returns 0 or JPEG_STATUS_CORRUPT; after an error the
// remaining blocks are zero.
__host__ __device__ inline int jpeg_entropy_file(const uint8_t* file, const JpegDesc& d, int16_t* coef, JpegHuff* tabs) {
    const int nc = d.ncomp;
    for (int c = 0; c < nc; ++c) {
        jpeg_build_huff(jpeg_table_bytes(file, d.dc[c]), tabs[2 * c]);
        jpeg_build_huff(jpeg_table_bytes(file, d.ac[c]), tabs[2 * c + 1]);
    }
    const int bpm = nc == 1 ? 1 : d.hs * d.vs;          // luma blocks per MCU
    const int lbw = d.mcux * (nc == 1 ? 1 : d.hs);      // luma plane width in blocks
    const int64_t lplane = (int64_t)lbw * d.mcuy * (nc == 1 ? 1 : d.vs);
    const int64_t cplane = (int64_t)d.mcux * d.mcuy;
    JpegBits br{file, d.scan, d.scan_end, 0, 0, 0, false};
    int pred[3] = {0, 0, 0};
    int next_rst = 0;
    bool bad = false;
    const int64_t total = (int64_t)d.mcux * d.mcuy;
    int64_t left = d.ri;
    for (int64_t mcu = 0; mcu < total; ++mcu) {
        if (d.ri && left == 0) {                         // restart: drop the buffered bits, expect RST(next_rst), reset the predictors
            if (!bad) {
                int64_t q = br.pos;
                while (q < br.end && file[q] == 0xFF) ++q;
                if (q >= br.end || q == br.pos || file[q] != 0xD0 + next_rst) bad = true;
                else br.pos = q + 1;
            }
            br.buf = 0; br.nbits = 0; br.pad = 0; br.marker = false;
            pred[0] = pred[1] = pred[2] = 0;
            next_rst = (next_rst + 1) & 7;
            left = d.ri;
        }
        --left;
        const int mx = (int)(mcu % d.mcux), my = (int)(mcu / d.mcux);
        for (int blk = 0; blk < bpm + (nc == 1 ? 0 : 2); ++blk) {
            int c;
            int16_t* out;
            if (blk < bpm) {
                c = 0;
                const int bx = mx * (nc == 1 ? 1 : d.hs) + (nc == 1 ? 0 : blk % d.hs);
                const int by = my * (nc == 1 ? 1 : d.vs) + (nc == 1 ? 0 : blk / d.hs);
                out = coef + ((int64_t)by * lbw + bx) * 64;
            } else {
                c = blk - bpm + 1;
                out = coef + (lplane + (c - 1) * cplane + (int64_t)my * d.mcux + mx) * 64;
            }
            for (int k = 0; k < 64; ++k) out[k] = 0;
            if (bad) continue;
            br.fill();
            int s = jpeg_decode_sym(br, tabs[2 * c], bad);
            if (s) {
                br.fill();
                const int r = (int)br.peek(s);
                br.skip(s);
                s = jpeg_extend(r, s);
            }
            pred[c] += s;
            out[0] = (int16_t)pred[c];
            const JpegHuff& ac = tabs[2 * c + 1];
            for (int k = 1; k < 64; ++k) {
                br.fill();
                int rs = jpeg_decode_sym(br, ac, bad);
                const int r = rs >> 4;
                s = rs & 15;
                if (s) {
                    k += r;
                    const int v = (int)br.peek(s);
                    br.skip(s);
                    out[jpeg_natural(k)] = (int16_t)jpeg_extend(v, s);
                } else {
                    if (r != 15) break;
                    k += 15;
                }
            }
            if (bad || br.overrun()) { bad = true; for (int k = 0; k < 64; ++k) out[k] = 0; }
        }
    }
    return bad ? JPEG_STATUS_CORRUPT : 0;
}

// ---------------------------------------------------------------------------------------------------------------------------------
// stage 2: dequantisation + jpeg_idct_islow (jidctint.c), the range-limit table of jdmaster.c indexed with & RANGE_MASK
// ---------------------------------------------------------------------------------------------------------------------------------
__host__ __device__ inline uint8_t jpeg_range_limit(int v) {      // IDCT_range_limit(cinfo)[v & 1023]
    const int x = v & 1023;
    return x < 128 ? (uint8_t)(x + 128) : x < 512 ? (uint8_t)255 : x < 896 ? (uint8_t)0 : (uint8_t)(x - 896);
}

#define YF_IDCT_BODY(i0, i1, i2, i3, i4, i5, i6, i7)                                                                                   \
    int64_t z1, z2, z3, z4, z5, tmp0, tmp1, tmp2, tmp3, tmp10, tmp11, tmp12, tmp13;                                                     \
    z2 = (i2); z3 = (i6);                                                                                                              \
    z1 = (z2 + z3) * 4433;                                                                                                             \
    tmp2 = z1 + z3 * -15137;                                                                                                           \
    tmp3 = z1 + z2 * 6270;                                                                                                             \
    z2 = (i0); z3 = (i4);                                                                                                              \
    tmp0 = (z2 + z3) * 8192;                                                                                                           \
    tmp1 = (z2 - z3) * 8192;                                                                                                           \
    tmp10 = tmp0 + tmp3; tmp13 = tmp0 - tmp3; tmp11 = tmp1 + tmp2; tmp12 = tmp1 - tmp2;                                               \
    tmp0 = (i7); tmp1 = (i5); tmp2 = (i3); tmp3 = (i1);                                                                                \
    z1 = tmp0 + tmp3; z2 = tmp1 + tmp2; z3 = tmp0 + tmp2; z4 = tmp1 + tmp3;                                                            \
    z5 = (z3 + z4) * 9633;                                                                                                             \
    tmp0 = tmp0 * 2446; tmp1 = tmp1 * 16819; tmp2 = tmp2 * 25172; tmp3 = tmp3 * 12299;                                                \
    z1 = z1 * -7373; z2 = z2 * -20995; z3 = z3 * -16069; z4 = z4 * -3196;                                                              \
    z3 += z5; z4 += z5;                                                                                                                \
    tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;

// coef: 64 quantised coefficients (natural order); q: 64 quantisation values (natural order); out: 8 rows of 8 samples, row pitch 8
__host__ __device__ inline void jpeg_idct_islow(const int16_t* coef, const int32_t* q, uint8_t* out) {
    int ws[64];
#pragma unroll
    for (int c = 0; c < 8; ++c) {                        // pass 1: columns, results scaled by 2^PASS1_BITS
        const int16_t* in = coef + c;
        const int32_t* qq = q + c;
        if (!in[8] && !in[16] && !in[24] && !in[32] && !in[40] && !in[48] && !in[56]) {
            const int dc = (in[0] * qq[0]) * 4;
            for (int r = 0; r < 8; ++r) ws[r * 8 + c] = dc;
            continue;
        }
        YF_IDCT_BODY((int64_t)in[0] * qq[0], (int64_t)in[8] * qq[8], (int64_t)in[16] * qq[16], (int64_t)in[24] * qq[24],
                     (int64_t)in[32] * qq[32], (int64_t)in[40] * qq[40], (int64_t)in[48] * qq[48], (int64_t)in[56] * qq[56])
        ws[0 * 8 + c] = (int)((tmp10 + tmp3 + (1 << 10)) >> 11);
        ws[7 * 8 + c] = (int)((tmp10 - tmp3 + (1 << 10)) >> 11);
        ws[1 * 8 + c] = (int)((tmp11 + tmp2 + (1 << 10)) >> 11);
        ws[6 * 8 + c] = (int)((tmp11 - tmp2 + (1 << 10)) >> 11);
        ws[2 * 8 + c] = (int)((tmp12 + tmp1 + (1 << 10)) >> 11);
        ws[5 * 8 + c] = (int)((tmp12 - tmp1 + (1 << 10)) >> 11);
        ws[3 * 8 + c] = (int)((tmp13 + tmp0 + (1 << 10)) >> 11);
        ws[4 * 8 + c] = (int)((tmp13 - tmp0 + (1 << 10)) >> 11);
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {                        // pass 2: rows, descaled by 2^(CONST_BITS + PASS1_BITS + 3)
        const int* w = ws + r * 8;
        uint8_t* o = out + r * 8;
        if (!w[1] && !w[2] && !w[3] && !w[4] && !w[5] && !w[6] && !w[7]) {
            const uint8_t v = jpeg_range_limit((int)(((int64_t)w[0] + (1 << 4)) >> 5));
            for (int c = 0; c < 8; ++c) o[c] = v;
            continue;
        }
        YF_IDCT_BODY((int64_t)w[0], (int64_t)w[1], (int64_t)w[2], (int64_t)w[3], (int64_t)w[4], (int64_t)w[5], (int64_t)w[6], (int64_t)w[7])
        o[0] = jpeg_range_limit((int)((tmp10 + tmp3 + (1 << 17)) >> 18));
        o[7] = jpeg_range_limit((int)((tmp10 - tmp3 + (1 << 17)) >> 18));
        o[1] = jpeg_range_limit((int)((tmp11 + tmp2 + (1 << 17)) >> 18));
        o[6] = jpeg_range_limit((int)((tmp11 - tmp2 + (1 << 17)) >> 18));
        o[2] = jpeg_range_limit((int)((tmp12 + tmp1 + (1 << 17)) >> 18));
        o[5] = jpeg_range_limit((int)((tmp12 - tmp1 + (1 << 17)) >> 18));
        o[3] = jpeg_range_limit((int)((tmp13 + tmp0 + (1 << 17)) >> 18));
        o[4] = jpeg_range_limit((int)((tmp13 - tmp0 + (1 << 17)) >> 18));
    }
}

// component c's quantisation table in natural order
__host__ __device__ inline void jpeg_quant(const uint8_t* file, const JpegDesc& d, int c, int32_t* q) {
    const uint8_t* t = file + d.q[c];
    const bool wide = (d.qprec >> c) & 1;
    for (int i = 0; i < 64; ++i) q[jpeg_natural(i)] = wide ? (t[2 * i] << 8) | t[2 * i + 1] : t[i];
}

// ---------------------------------------------------------------------------------------------------------------------------------
// stage 3: upsampling (jdsample.c) + colour conversion (jdcolor.c). `smp` = the file's blocks after stage 2: block i's samples are the
// first 64 bytes of its 128.
// ---------------------------------------------------------------------------------------------------------------------------------
__host__ __device__ inline int jpeg_sample(const uint8_t* smp, int64_t plane, int bw, int x, int y) {
    return smp[(plane + (int64_t)(y >> 3) * bw + (x >> 3)) * 128 + (y & 7) * 8 + (x & 7)];
}

// chroma sample of component plane `plane` (bw blocks wide) at output pixel (x, y)
__host__ __device__ inline int jpeg_chroma(const uint8_t* smp, const JpegDesc& d, int64_t plane, int bw, int x, int y) {
    if (d.hs == 1) return jpeg_sample(smp, plane, bw, x, y);
    const int dw = (d.w + 1) >> 1;                       // downsampled_width = ceil(w / 2)
    const int cx = x >> 1;
    if (dw <= 2) return jpeg_sample(smp, plane, bw, cx, d.vs == 2 ? y >> 1 : y);   // plain replication (fancy needs width > 2)
    const bool odd = x & 1;
    const bool edge = odd ? cx == dw - 1 : cx == 0;
    const int nx = odd ? cx + 1 : cx - 1;
    if (d.vs == 1) {                                     // h2v1_fancy_upsample
        const int a = jpeg_sample(smp, plane, bw, cx, y);
        if (edge) return a;
        return (3 * a + jpeg_sample(smp, plane, bw, nx, y) + (odd ? 2 : 1)) >> 2;
    }
    const int dh = (d.h + 1) >> 1;                       // h2v2_fancy_upsample: the rows above / below clamp to the image
    const int cy = y >> 1;
    int fy = (y & 1) ? cy + 1 : cy - 1;
    fy = fy < 0 ? 0 : fy > dh - 1 ? dh - 1 : fy;
    const int t = 3 * jpeg_sample(smp, plane, bw, cx, cy) + jpeg_sample(smp, plane, bw, cx, fy);
    if (edge) return odd ? (t * 4 + 7) >> 4 : (t * 4 + 8) >> 4;
    const int u = 3 * jpeg_sample(smp, plane, bw, nx, cy) + jpeg_sample(smp, plane, bw, nx, fy);
    return odd ? (t * 3 + u + 7) >> 4 : (t * 3 + u + 8) >> 4;
}

__host__ __device__ inline uint8_t jpeg_clamp(int v) { return (uint8_t)(v < 0 ? 0 : v > 255 ? 255 : v); }

// BGR of output pixel (x, y)
__host__ __device__ inline void jpeg_pixel(const uint8_t* smp, const JpegDesc& d, int x, int y, uint8_t* bgr) {
    if (d.ncomp == 1) {
        const uint8_t g = (uint8_t)jpeg_sample(smp, 0, d.mcux, x, y);
        bgr[0] = bgr[1] = bgr[2] = g;
        return;
    }
    const int lbw = d.mcux * d.hs;
    const int64_t lplane = (int64_t)lbw * d.mcuy * d.vs, cplane = (int64_t)d.mcux * d.mcuy;
    const int Y = jpeg_sample(smp, 0, lbw, x, y);
    const int cb = jpeg_chroma(smp, d, lplane, d.mcux, x, y) - 128;
    const int cr = jpeg_chroma(smp, d, lplane + cplane, d.mcux, x, y) - 128;
    // build_ycc_rgb_table, SCALEBITS 16: FIX(1.40200) = 91881, FIX(1.77200) = 116130, FIX(0.71414) = 46802, FIX(0.34414) = 22554
    const int r = (int)((91881LL * cr + 32768) >> 16);
    const int b = (int)((116130LL * cb + 32768) >> 16);
    const int g = (int)((-46802LL * cr + (-22554LL * cb + 32768)) >> 16);
    bgr[0] = jpeg_clamp(Y + b);
    bgr[1] = jpeg_clamp(Y + g);
    bgr[2] = jpeg_clamp(Y + r);
}

// ---------------------------------------------------------------------------------------------------------------------------------
// kernels (one launch of each per chunk of JPEG_CHUNK files)
// ---------------------------------------------------------------------------------------------------------------------------------
// FPW files per warp: 1 (lane 0 of each 32-thread block decodes one file) or 32 (one file per lane). Each file has 6 Huffman tables of
// shared memory.
constexpr int JPEG_TABS_BYTES = 6 * (int)sizeof(JpegHuff);
template <int FPW>
__global__ void __launch_bounds__(32)
jpeg_entropy_kernel(const uint8_t* __restrict__ files, const __grid_constant__ JpegChunk ch, int n, int16_t* __restrict__ coef,
                    int32_t* __restrict__ status) {
    extern __shared__ __align__(16) unsigned char jpeg_smem[];
    const int slot = FPW == 1 ? 0 : threadIdx.x;
    const int i = blockIdx.x * FPW + slot;
    if (FPW == 1 && threadIdx.x != 0) return;
    if (i >= n) return;
    const JpegDesc& d = ch.d[i];
    JpegHuff* tabs = reinterpret_cast<JpegHuff*>(jpeg_smem) + slot * 6;
    status[i] = jpeg_entropy_file(files + d.src, d, coef + d.cbase * 64, tabs);
}

constexpr int JPEG_IDCT_NT = 128;
__global__ void __launch_bounds__(JPEG_IDCT_NT)
jpeg_idct_kernel(const uint8_t* __restrict__ files, const __grid_constant__ JpegChunk ch, int16_t* __restrict__ coef) {
    __shared__ int32_t q[3][64];
    const JpegDesc& d = ch.d[blockIdx.y];
    for (int t = threadIdx.x; t < d.ncomp * 64; t += JPEG_IDCT_NT) {
        const int c = t >> 6, i = t & 63;
        const uint8_t* tb = files + d.src + d.q[c];
        q[c][jpeg_natural(i)] = ((d.qprec >> c) & 1) ? (tb[2 * i] << 8) | tb[2 * i + 1] : tb[i];
    }
    __syncthreads();
    const int64_t nb = jpeg_blocks(d);
    const int64_t lplane = d.ncomp == 1 ? nb : (int64_t)d.mcux * d.hs * d.mcuy * d.vs;
    const int64_t cplane = (int64_t)d.mcux * d.mcuy;
    int16_t* base = coef + d.cbase * 64;
    for (int64_t b = blockIdx.x * (int64_t)JPEG_IDCT_NT + threadIdx.x; b < nb; b += (int64_t)gridDim.x * JPEG_IDCT_NT) {
        const int c = b < lplane ? 0 : b < lplane + cplane ? 1 : 2;
        int16_t blk[64];
        const uint4* src = reinterpret_cast<const uint4*>(base + b * 64);
#pragma unroll
        for (int k = 0; k < 8; ++k) reinterpret_cast<uint4*>(blk)[k] = src[k];
        uint8_t out[64];
        jpeg_idct_islow(blk, q[c], out);
        uint4* dst = reinterpret_cast<uint4*>(base + b * 64);
#pragma unroll
        for (int k = 0; k < 4; ++k) dst[k] = reinterpret_cast<const uint4*>(out)[k];
    }
}

constexpr int JPEG_COLOR_NT = 256;
__global__ void __launch_bounds__(JPEG_COLOR_NT)
jpeg_color_kernel(const __grid_constant__ JpegChunk ch, const int16_t* __restrict__ coef, uint8_t* __restrict__ frames) {
    const JpegDesc& d = ch.d[blockIdx.y];
    const uint8_t* smp = reinterpret_cast<const uint8_t*>(coef + d.cbase * 64);
    const int64_t npx = (int64_t)d.h * d.w;
    uint8_t* out = frames + d.dst;
    for (int64_t p = blockIdx.x * (int64_t)JPEG_COLOR_NT + threadIdx.x; p < npx; p += (int64_t)gridDim.x * JPEG_COLOR_NT) {
        const int y = (int)(p / d.w), x = (int)(p % d.w);
        uint8_t bgr[3];
        jpeg_pixel(smp, d, x, y, bgr);
        out[p * 3 + 0] = bgr[0];
        out[p * 3 + 1] = bgr[1];
        out[p * 3 + 2] = bgr[2];
    }
}

}  // namespace yf
