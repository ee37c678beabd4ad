// yf_jpeg_enc.cuh — baseline JPEG encoding on the device, byte-identical to cv2.imencode(".jpg", frame, [IMWRITE_JPEG_QUALITY, q,
// IMWRITE_JPEG_SAMPLING_FACTOR, s]) (libjpeg-turbo with OpenCV's settings: JDCT_ISLOW, standard Huffman tables, no restart
// intervals, JFIF 1.01 APP0). DESIGN.md §5.8.
//
//   host    jpeg_enc_header: SOI .. SOS for (h, w, quality, sampling) (jcmarker.c), jpeg_enc_qtables (jcparam.c), jpeg_enc_bound.
//   kernel  jpeg_enc_dct_kernel: 8 threads per 8x8 block, blocks in MCU-interleaved scan order: BGR -> YCbCr (jccolor.c), edge
//           replication and h2v1 / h2v2 downsampling (jcprepct.c, jcsample.c), jpeg_fdct_islow (jfdctint.c), quantisation
//           (jcdctmgr.c); dummy blocks of a partial MCU (jccoefct.c) are zero with the DC of the block they copy. int16 coefficients,
//           zigzag order.
//   kernel  jpeg_enc_len_kernel: one 512-thread block per file: each block's Huffman bit length (jchuff.c) from its coefficients and
//           the DC of the previous block of its component, an exclusive scan of the lengths (each thread sums a contiguous run of
//           blocks), and the file's bit buffer zeroed up to its length.
//   kernel  jpeg_enc_emit_kernel: one thread per block writes its codes MSB-first at its bit offset; 32-bit words are ORed in with
//           atomicOr (neighbouring blocks share their boundary words). The file's last block adds the 1-bit padding.
//   kernel  jpeg_enc_stuff_kernel: one 512-thread block per file: the header bytes, then the scan bytes in tiles of 16 bytes a
//           thread, each tile's 0xFF count scanned across the block so that every byte lands at its stuffed position with a 0x00
//           after each 0xFF, then EOI and the file's length.
//
// The per-block arithmetic is __host__ __device__ so that it can be checked against cv2 on a machine without a GPU; the library itself
// only ever runs it on the device.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstring>

#include "yf_jpeg.cuh"

namespace yf {

constexpr int JPEG_ENC_CHUNK = 256;                     // frames per launch: 256 x 56 bytes of descriptors + 256 bytes of divisors
constexpr int JPEG_ENC_SAMPLING_420 = 0x221111;         // cv2.IMWRITE_JPEG_SAMPLING_FACTOR_* (YF_JPEG_SAMPLING_*)
constexpr int JPEG_ENC_SAMPLING_422 = 0x211111;
constexpr int JPEG_ENC_SAMPLING_444 = 0x111111;
constexpr int JPEG_ENC_HEADER_BYTES = 623;              // SOI, APP0, 2 DQT, SOF0, 4 DHT, SOS of a 3-component file

struct JpegEncDesc {
    int64_t src;                // offset of the BGR frame in the frames buffer
    int64_t dst;                // offset of the file in the output buffer
    int64_t cbase;              // first block of the frame in the coefficient workspace (relative to the chunk)
    int64_t bbase;              // first byte of the frame's bit buffer in the workspace (relative to the chunk), a multiple of 16
    int32_t hdr;                // offset of the frame's header bytes in the staged headers
    int32_t hdr_len;
    uint16_t h, w;
    uint16_t mcux, mcuy;        // MCUs per row / column
    uint8_t hs, vs;             // luma sampling factors (chroma 1x1)
    uint8_t pad[6];
};
static_assert(sizeof(JpegEncDesc) == 56, "JpegEncDesc layout");
struct JpegEncChunk {
    JpegEncDesc d[JPEG_ENC_CHUNK];
    uint16_t qdiv[2][64];       // quantisation divisors (table << 3, jcdctmgr.c for JDCT_ISLOW), luma / chroma, natural order
};

// Huffman codes of the standard tables (jchuff.c jpeg_make_c_derived_tbl over jstdhuff.c): e[t][symbol] = (length << 16) | code,
// t = 0 DC luma, 1 AC luma, 2 DC chroma, 3 AC chroma
struct JpegEncTabs { uint32_t e[4][256]; };
constexpr JpegEncTabs jpeg_enc_make_tabs() {
    constexpr uint8_t std_tabs[412] = YF_JPEG_STD_TABLES;
    constexpr int base[4] = {0, 28, 206, 234};
    JpegEncTabs t{};
    for (int k = 0; k < 4; ++k) {
        int p = 0;
        uint32_t code = 0;
        for (int l = 1; l <= 16; ++l) {
            for (int i = 0; i < std_tabs[base[k] + l - 1]; ++i, ++p, ++code) t.e[k][std_tabs[base[k] + 16 + p]] = ((uint32_t)l << 16) | code;
            code <<= 1;
        }
    }
    return t;
}
static constexpr JpegEncTabs h_jpeg_enc_tabs = jpeg_enc_make_tabs();
__constant__ JpegEncTabs c_jpeg_enc_tabs = jpeg_enc_make_tabs();

// most bits one block can take: the longest DC code + category 11, then 63 coefficients of at most the longest AC code + 10 bits
// (a run / ZRL / EOB code stands for one or more zero coefficients and is no longer than that)
inline int jpeg_enc_block_max_bits() {
    int dc = 0, ac = 0;
    for (int t = 0; t < 4; ++t)
        for (int s = 0; s < 256; ++s) {
            const uint32_t e = h_jpeg_enc_tabs.e[t][s];
            if (!e) continue;
            const int bits = (int)(e >> 16) + (s & 15);
            if (t & 1) ac = bits > ac ? bits : ac;
            else dc = bits > dc ? bits : dc;
        }
    return dc + 63 * ac;
}

// ---------------------------------------------------------------------------------------------------------------------------------
// host: parameters, tables, header bytes, bounds
// ---------------------------------------------------------------------------------------------------------------------------------
inline bool jpeg_enc_sampling(int sampling, int& hs, int& vs) {
    switch (sampling) {
        case JPEG_ENC_SAMPLING_420: hs = 2; vs = 2; return true;
        case JPEG_ENC_SAMPLING_422: hs = 2; vs = 1; return true;
        case JPEG_ENC_SAMPLING_444: hs = 1; vs = 1; return true;
        default: return false;
    }
}

__host__ __device__ inline int64_t jpeg_enc_blocks(int h, int w, int hs, int vs) {
    const int64_t mcux = (w + 8 * hs - 1) / (8 * hs), mcuy = (h + 8 * vs - 1) / (8 * vs);
    return mcux * mcuy * (hs * vs + 2);
}

// jpeg_set_quality(q, force_baseline = TRUE): tables of ITU-T T.81 K.1 scaled, in zigzag order (the order of DQT and of the divisors)
inline void jpeg_enc_qtables(int quality, int qz[2][64]) {
    static const uint8_t base[2][64] = {
        {16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22, 29, 51, 87, 80, 62,
         18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, 49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99},
        {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99,
         99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99}};
    const int scale = quality < 50 ? 5000 / quality : 200 - 2 * quality;
    for (int t = 0; t < 2; ++t)
        for (int k = 0; k < 64; ++k) {
            const int v = ((int)base[t][h_jpeg_natural[k]] * scale + 50) / 100;
            qz[t][k] = v < 1 ? 1 : v > 255 ? 255 : v;
        }
}

// SOI .. SOS as libjpeg-turbo writes them for cv2 (jcmarker.c): APP0 JFIF 1.01 (no density unit, 1:1, no thumbnail), one DQT segment
// per table, SOF0, the DHT segments DC0 AC0 DC1 AC1, SOS. Returns JPEG_ENC_HEADER_BYTES.
inline int jpeg_enc_header(int h, int w, int quality, int hs, int vs, uint8_t* out) {
    int qz[2][64];
    jpeg_enc_qtables(quality, qz);
    uint8_t* p = out;
    auto put = [&](std::initializer_list<int> bytes) { for (int b : bytes) *p++ = (uint8_t)b; };
    put({0xFF, 0xD8, 0xFF, 0xE0, 0, 16, 'J', 'F', 'I', 'F', 0, 1, 1, 0, 0, 1, 0, 1, 0, 0});
    for (int t = 0; t < 2; ++t) {
        put({0xFF, 0xDB, 0, 67, t});
        for (int k = 0; k < 64; ++k) *p++ = (uint8_t)qz[t][k];
    }
    put({0xFF, 0xC0, 0, 17, 8, h >> 8, h & 255, w >> 8, w & 255, 3, 1, (hs << 4) | vs, 0, 2, 0x11, 1, 3, 0x11, 1});
    static const int off[4] = {0, 28, 206, 234}, cls[4] = {0x00, 0x10, 0x01, 0x11};
    for (int t = 0; t < 4; ++t) {
        const uint8_t* tab = h_jpeg_std + off[t];
        int n = 0;
        for (int l = 0; l < 16; ++l) n += tab[l];
        put({0xFF, 0xC4, (19 + n) >> 8, (19 + n) & 255, cls[t]});
        memcpy(p, tab, 16 + n);
        p += 16 + n;
    }
    put({0xFF, 0xDA, 0, 12, 3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0});
    return (int)(p - out);
}

// most bytes of the entropy-coded data of one frame before stuffing, and of one whole file (headers + every byte stuffed + EOI)
inline int64_t jpeg_enc_scan_max(int h, int w, int hs, int vs) {
    return (jpeg_enc_blocks(h, w, hs, vs) * jpeg_enc_block_max_bits() + 7) / 8;
}
inline int64_t jpeg_enc_file_max(int h, int w, int hs, int vs) { return JPEG_ENC_HEADER_BYTES + 2 * jpeg_enc_scan_max(h, w, hs, vs) + 2; }

// ---------------------------------------------------------------------------------------------------------------------------------
// stage 1: colour conversion, downsampling, forward DCT, quantisation
// ---------------------------------------------------------------------------------------------------------------------------------
// rgb_ycc_convert (jccolor.c), SCALEBITS 16: FIX(0.29900) = 19595, FIX(0.58700) = 38470, FIX(0.11400) = 7471, FIX(0.16874) = 11059,
// FIX(0.33126) = 21709, FIX(0.5) = 32768, FIX(0.41869) = 27439, FIX(0.08131) = 5329; chroma rounds with ONE_HALF - 1
__host__ __device__ inline int jpeg_enc_ycc(const uint8_t* px, int c) {
    const int b = px[0], g = px[1], r = px[2];
    if (c == 0) return (19595 * r + 38470 * g + 7471 * b + 32768) >> 16;
    if (c == 1) return (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16;
    return (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16;
}

__host__ __device__ inline int jpeg_enc_px(const uint8_t* f, int w, int x, int y, int c) { return jpeg_enc_ycc(f + ((int64_t)y * w + x) * 3, c); }

// Row r of block (bx, by) of component c (component sample coordinates) -> its 8 samples - 128. Columns past the image repeat its last
// column before downsampling (expand_right_edge); rows past it repeat its last row, and at 4:2:0 the chroma rows below the last real
// one repeat that row (expand_bottom_edge of the downsampled rows, jcprepct.c). h2v1 averages with biases 0, 1 alternating, h2v2
// with 1, 2 (jcsample.c).
__host__ __device__ inline void jpeg_enc_row(const uint8_t* f, const JpegEncDesc& d, int c, int bx, int by, int r, int* o) {
    const int h = d.h, w = d.w, y = by * 8 + r;
    if (c == 0 || d.hs == 1) {
        const int yy = y < h ? y : h - 1;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int x = bx * 8 + k;
            o[k] = jpeg_enc_px(f, w, x < w ? x : w - 1, yy, c) - 128;
        }
    } else if (d.vs == 1) {
        const int yy = y < h ? y : h - 1;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int x = 2 * (bx * 8 + k);
            const int xa = x < w ? x : w - 1, xb = x + 1 < w ? x + 1 : w - 1;
            o[k] = ((jpeg_enc_px(f, w, xa, yy, c) + jpeg_enc_px(f, w, xb, yy, c) + (k & 1)) >> 1) - 128;
        }
    } else {
        const int ch = (h + 1) >> 1;
        const int yy = y < ch ? y : ch - 1;
        const int ya = 2 * yy, yb = 2 * yy + 1 < h ? 2 * yy + 1 : h - 1;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int x = 2 * (bx * 8 + k);
            const int xa = x < w ? x : w - 1, xb = x + 1 < w ? x + 1 : w - 1;
            o[k] = ((jpeg_enc_px(f, w, xa, ya, c) + jpeg_enc_px(f, w, xb, ya, c) + jpeg_enc_px(f, w, xa, yb, c) +
                     jpeg_enc_px(f, w, xb, yb, c) + 1 + (k & 1)) >> 2) - 128;
        }
    }
}

// jpeg_fdct_islow (jfdctint.c), CONST_BITS 13, PASS1_BITS 2: one 8-point pass in place on v[0], v[s], .., v[7 s]. Pass 1 (rows)
// scales up by 2^PASS1_BITS, pass 2 (columns) descales; the outputs are the DCT scaled by 8. 32-bit arithmetic suffices for 8-bit
// samples (jfdctint.c).
template <int PASS>
__host__ __device__ inline void jpeg_fdct_pass(int* v, int s) {
    const int tmp0 = v[0] + v[7 * s], tmp7 = v[0] - v[7 * s], tmp1 = v[s] + v[6 * s], tmp6 = v[s] - v[6 * s];
    const int tmp2 = v[2 * s] + v[5 * s], tmp5 = v[2 * s] - v[5 * s], tmp3 = v[3 * s] + v[4 * s], tmp4 = v[3 * s] - v[4 * s];
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    constexpr int D = PASS == 1 ? 11 : 15;              // CONST_BITS -/+ PASS1_BITS
    v[0] = PASS == 1 ? (tmp10 + tmp11) * 4 : (tmp10 + tmp11 + 2) >> 2;
    v[4 * s] = PASS == 1 ? (tmp10 - tmp11) * 4 : (tmp10 - tmp11 + 2) >> 2;
    const int z1 = (tmp12 + tmp13) * 4433;
    v[2 * s] = (z1 + tmp13 * 6270 + (1 << (D - 1))) >> D;
    v[6 * s] = (z1 - tmp12 * 15137 + (1 << (D - 1))) >> D;
    const int z5 = (tmp4 + tmp5 + tmp6 + tmp7) * 9633;
    const int a1 = (tmp4 + tmp7) * -7373, a2 = (tmp5 + tmp6) * -20995;
    const int a3 = (tmp4 + tmp6) * -16069 + z5, a4 = (tmp5 + tmp7) * -3196 + z5;
    v[7 * s] = (tmp4 * 2446 + a1 + a3 + (1 << (D - 1))) >> D;
    v[5 * s] = (tmp5 * 16819 + a2 + a4 + (1 << (D - 1))) >> D;
    v[3 * s] = (tmp6 * 25172 + a2 + a3 + (1 << (D - 1))) >> D;
    v[1 * s] = (tmp7 * 12299 + a1 + a4 + (1 << (D - 1))) >> D;
}

// quantisation (jcdctmgr.c): (|x| + q / 2) / q with the sign of x, q = table << 3
__host__ __device__ inline int16_t jpeg_enc_quant(int v, int q) {
    const int a = ((v < 0 ? -v : v) + (q >> 1)) / q;
    return (int16_t)(v < 0 ? -a : a);
}

// Block i of the frame's scan (MCU-interleaved: hs*vs luma blocks row by row, then Cb, then Cr) -> component c and the block whose
// samples it codes (bx, by); `dummy` when the block lies past the luma plane's blocks: it is coded as zero with the DC of the block
// compress_data copies (the last real block of its MCU row, or of the MCU's first row when its own row is past the plane).
__host__ __device__ inline void jpeg_enc_block_pos(const JpegEncDesc& d, int64_t i, int& c, int& bx, int& by, bool& dummy) {
    const int L = d.hs * d.vs;
    const int64_t mcu = i / (L + 2);
    const int k = (int)(i - mcu * (L + 2));
    const int mx = (int)(mcu % d.mcux), my = (int)(mcu / d.mcux);
    dummy = false;
    if (k >= L) { c = k - L + 1; bx = mx; by = my; return; }
    c = 0;
    const int row = k / d.hs, col = k - row * d.hs;
    const int wib = (d.w + 7) >> 3, hib = (d.h + 7) >> 3;
    bx = mx * d.hs + col;
    by = my * d.vs + row;
    if (bx < wib && by < hib) return;
    dummy = true;
    const int last = wib - 1 - mx * d.hs < d.hs - 1 ? wib - 1 - mx * d.hs : d.hs - 1;
    bx = mx * d.hs + last;
    if (by >= hib) by = my * d.vs;
}

// ---------------------------------------------------------------------------------------------------------------------------------
// stages 2 and 4: Huffman coding of one block (encode_one_block, jchuff.c) into a sink: a bit counter or a bit writer
// ---------------------------------------------------------------------------------------------------------------------------------
__host__ __device__ inline int jpeg_enc_cat(int v) {
    const unsigned a = (unsigned)(v < 0 ? -v : v);
#ifdef __CUDA_ARCH__
    return 32 - __clz(a);
#else
    return a ? 32 - __builtin_clz(a) : 0;
#endif
}

// index of the block before block i of the same component in scan order, -1 for the first one (the DC predictors start at 0)
__host__ __device__ inline int64_t jpeg_enc_prev(const JpegEncDesc& d, int64_t i) {
    const int L = d.hs * d.vs;
    const int k = (int)(i % (L + 2));
    return k >= L ? i - (L + 2) : k > 0 ? i - 1 : i - 3;
}

template <class Sink>
__host__ __device__ inline void jpeg_enc_code_block(const int16_t* zz, int prev_dc, const uint32_t* dct, const uint32_t* act, Sink& out) {
    int v = zz[0] - prev_dc;
    int s = jpeg_enc_cat(v);
    out.put(((dct[s] & 0xFFFF) << s) | ((uint32_t)(v < 0 ? v - 1 : v) & ((1u << s) - 1)), (int)(dct[s] >> 16) + s);
    int r = 0;
    for (int k = 1; k < 64; ++k) {
        v = zz[k];
        if (!v) { ++r; continue; }
        for (; r > 15; r -= 16) out.put(act[0xF0] & 0xFFFF, (int)(act[0xF0] >> 16));
        s = jpeg_enc_cat(v);
        const uint32_t e = act[(r << 4) + s];
        out.put(((e & 0xFFFF) << s) | ((uint32_t)(v < 0 ? v - 1 : v) & ((1u << s) - 1)), (int)(e >> 16) + s);
        r = 0;
    }
    if (r) out.put(act[0] & 0xFFFF, (int)(act[0] >> 16));
}

struct JpegBitCount {
    int64_t n = 0;
    __host__ __device__ void put(uint32_t, int len) { n += len; }
};

// MSB-first writer from bit `pos` of a zeroed buffer: words are ORed in (atomically on the device), so that blocks sharing a word
// may write it in any order. Values of at most 27 bits.
struct JpegBitWriter {
    uint32_t* words;
    int64_t w;
    uint64_t acc = 0;
    int fill;
    __host__ __device__ JpegBitWriter(uint32_t* words_, int64_t pos) : words(words_), w(pos >> 5), fill((int)(pos & 31)) {}
    __host__ __device__ void word(uint32_t x) {         // x holds 4 stream bytes, first byte in its top bits
#ifdef __CUDA_ARCH__
        atomicOr(words + w, __byte_perm(x, 0, 0x0123));
#else
        words[w] |= __builtin_bswap32(x);
#endif
    }
    __host__ __device__ void put(uint32_t v, int len) {
        acc |= (uint64_t)v << (64 - fill - len);
        fill += len;
        if (fill >= 32) { word((uint32_t)(acc >> 32)); ++w; acc <<= 32; fill -= 32; }
    }
    __host__ __device__ void finish() { if (fill > 0) word((uint32_t)(acc >> 32)); }
};

// ---------------------------------------------------------------------------------------------------------------------------------
// kernels (one launch of each per chunk of JPEG_ENC_CHUNK frames)
// ---------------------------------------------------------------------------------------------------------------------------------
// 8 threads per block: thread r builds row r and runs pass 1 on it, then (after an exchange through shared memory) pass 2 on column r
// and quantises it.
constexpr int JPEG_ENC_DCT_NT = 128;
#define YF_JPEG_ZIGZAG                                                                                                                 \
    {0,  1,  5,  6,  14, 15, 27, 28, 2,  4,  7,  13, 16, 26, 29, 42, 3,  8,  12, 17, 25, 30, 41, 43, 9,  11, 18, 24, 31, 40, 44, 53,  \
     10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38, 46, 51, 55, 60, 21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, 62, 63}
__constant__ uint8_t c_jpeg_zigzag[64] = YF_JPEG_ZIGZAG;   // natural index -> zigzag index
__global__ void __launch_bounds__(JPEG_ENC_DCT_NT)
jpeg_enc_dct_kernel(const uint8_t* __restrict__ frames, const __grid_constant__ JpegEncChunk ch, int16_t* __restrict__ coef) {
    __shared__ int ws[JPEG_ENC_DCT_NT / 8][64];
    const JpegEncDesc& d = ch.d[blockIdx.y];
    const int64_t nb = jpeg_enc_blocks(d.h, d.w, d.hs, d.vs);
    const int bl = threadIdx.x >> 3, r = threadIdx.x & 7;
    const unsigned grp = 0xFFu << (threadIdx.x & 24);
    for (int64_t i = blockIdx.x * (int64_t)(JPEG_ENC_DCT_NT / 8) + bl; i < nb; i += (int64_t)gridDim.x * (JPEG_ENC_DCT_NT / 8)) {
        int c, bx, by;
        bool dummy;
        jpeg_enc_block_pos(d, i, c, bx, by, dummy);
        int v[8];
        jpeg_enc_row(frames + d.src, d, c, bx, by, r, v);
        jpeg_fdct_pass<1>(v, 1);
#pragma unroll
        for (int k = 0; k < 8; ++k) ws[bl][r * 8 + k] = v[k];
        __syncwarp(grp);
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = ws[bl][k * 8 + r];
        __syncwarp(grp);
        jpeg_fdct_pass<2>(v, 1);
        const uint16_t* q = ch.qdiv[c ? 1 : 0];
        int16_t* o = coef + (d.cbase + i) * 64;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int n = k * 8 + r;
            o[c_jpeg_zigzag[n]] = dummy && n ? 0 : jpeg_enc_quant(v[k], q[n]);
        }
    }
}

__device__ inline void jpeg_enc_load_tabs(uint32_t (*tabs)[256]) {
    for (int t = threadIdx.x; t < 4 * 256; t += blockDim.x) tabs[t >> 8][t & 255] = c_jpeg_enc_tabs.e[t >> 8][t & 255];
    __syncthreads();
}

// exclusive scan of one int64 per thread across the block; `total` = the sum. sm holds NT / 32 values.
template <int NT>
__device__ inline int64_t jpeg_enc_block_scan(int64_t v, int64_t* sm, int64_t& total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int64_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) sm[wid] = x;
    __syncthreads();
    if (wid == 0) {
        int64_t s = lane < NT / 32 ? sm[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t y = __shfl_up_sync(0xFFFFFFFFu, s, o);
            if (lane >= o) s += y;
        }
        if (lane < NT / 32) sm[lane] = s;
    }
    __syncthreads();
    const int64_t before = (wid ? sm[wid - 1] : 0) + x - v;
    total = sm[NT / 32 - 1];
    __syncthreads();
    return before;
}

constexpr int JPEG_ENC_SCAN_NT = 512;
__global__ void __launch_bounds__(JPEG_ENC_SCAN_NT)
jpeg_enc_len_kernel(const __grid_constant__ JpegEncChunk ch, const int16_t* __restrict__ coef, int64_t* __restrict__ offs,
                    int64_t* __restrict__ fbits, uint32_t* __restrict__ bits) {
    __shared__ uint32_t tabs[4][256];
    __shared__ int64_t sm[JPEG_ENC_SCAN_NT / 32];
    jpeg_enc_load_tabs(tabs);
    const JpegEncDesc& d = ch.d[blockIdx.x];
    const int64_t nb = jpeg_enc_blocks(d.h, d.w, d.hs, d.vs);
    const int64_t per = (nb + JPEG_ENC_SCAN_NT - 1) / JPEG_ENC_SCAN_NT;
    const int64_t i0 = min(nb, threadIdx.x * per), i1 = min(nb, i0 + per);
    const int16_t* cb = coef + d.cbase * 64;
    int64_t* ob = offs + d.cbase;
    int64_t sum = 0;
    const int L = d.hs * d.vs;
    for (int64_t i = i0; i < i1; ++i) {
        const int64_t p = jpeg_enc_prev(d, i);
        const int c = (int)(i % (L + 2)) < L ? 0 : 1;
        JpegBitCount n;
        jpeg_enc_code_block(cb + i * 64, p < 0 ? 0 : cb[p * 64], tabs[2 * c], tabs[2 * c + 1], n);
        ob[i] = n.n;
        sum += n.n;
    }
    int64_t total;
    int64_t run = jpeg_enc_block_scan<JPEG_ENC_SCAN_NT>(sum, sm, total);
    for (int64_t i = i0; i < i1; ++i) {
        const int64_t b = ob[i];
        ob[i] = run;
        run += b;
    }
    if (threadIdx.x == 0) fbits[blockIdx.x] = total;
    uint32_t* wb = bits + d.bbase / 4;
    for (int64_t j = threadIdx.x, nw = (total + 31) / 32; j < nw; j += JPEG_ENC_SCAN_NT) wb[j] = 0;
}

constexpr int JPEG_ENC_EMIT_NT = 256;
__global__ void __launch_bounds__(JPEG_ENC_EMIT_NT)
jpeg_enc_emit_kernel(const __grid_constant__ JpegEncChunk ch, const int16_t* __restrict__ coef, const int64_t* __restrict__ offs,
                     const int64_t* __restrict__ fbits, uint32_t* __restrict__ bits) {
    __shared__ uint32_t tabs[4][256];
    jpeg_enc_load_tabs(tabs);
    const JpegEncDesc& d = ch.d[blockIdx.y];
    const int64_t nb = jpeg_enc_blocks(d.h, d.w, d.hs, d.vs);
    const int16_t* cb = coef + d.cbase * 64;
    const int L = d.hs * d.vs;
    for (int64_t i = blockIdx.x * (int64_t)JPEG_ENC_EMIT_NT + threadIdx.x; i < nb; i += (int64_t)gridDim.x * JPEG_ENC_EMIT_NT) {
        const int64_t p = jpeg_enc_prev(d, i);
        const int c = (int)(i % (L + 2)) < L ? 0 : 1;
        JpegBitWriter wr(bits + d.bbase / 4, offs[d.cbase + i]);
        jpeg_enc_code_block(cb + i * 64, p < 0 ? 0 : cb[p * 64], tabs[2 * c], tabs[2 * c + 1], wr);
        if (i == nb - 1) {                               // flush_bits: the last byte is filled with 1-bits
            const int pad = (int)(-fbits[blockIdx.y] & 7);
            if (pad) wr.put((1u << pad) - 1, pad);
        }
        wr.finish();
    }
}

constexpr int JPEG_ENC_STUFF_NT = 512;
__global__ void __launch_bounds__(JPEG_ENC_STUFF_NT)
jpeg_enc_stuff_kernel(const __grid_constant__ JpegEncChunk ch, const uint8_t* __restrict__ hdrs, const int64_t* __restrict__ fbits,
                      const uint8_t* __restrict__ scan, uint8_t* __restrict__ out, int64_t* __restrict__ len) {
    __shared__ int64_t sm[JPEG_ENC_STUFF_NT / 32];
    const JpegEncDesc& d = ch.d[blockIdx.x];
    uint8_t* o = out + d.dst;
    for (int j = threadIdx.x; j < d.hdr_len; j += JPEG_ENC_STUFF_NT) o[j] = hdrs[d.hdr + j];
    const int64_t nbytes = (fbits[blockIdx.x] + 7) >> 3;
    const uint8_t* s = scan + d.bbase;
    int64_t carry = d.hdr_len;                          // output position of scan byte 0 of the tile, stuffing before it included
    for (int64_t t0 = 0; t0 < nbytes; t0 += 16 * JPEG_ENC_STUFF_NT) {
        const int64_t p = t0 + 16 * threadIdx.x;
        const int n = (int)max((int64_t)0, min((int64_t)16, nbytes - p));
        __align__(16) uint8_t b[16];
        *reinterpret_cast<uint4*>(b) = n ? *reinterpret_cast<const uint4*>(s + p) : make_uint4(0, 0, 0, 0);
        int ff = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) ff += k < n && b[k] == 0xFF;
        int64_t tile_ff;
        int64_t q = carry + p + jpeg_enc_block_scan<JPEG_ENC_STUFF_NT>(ff, sm, tile_ff);
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            if (k >= n) break;
            o[q++] = b[k];
            if (b[k] == 0xFF) o[q++] = 0;
        }
        carry += tile_ff;
    }
    if (threadIdx.x == 0) {
        const int64_t end = carry + nbytes;
        o[end] = 0xFF;
        o[end + 1] = 0xD9;
        len[blockIdx.x] = end + 2;
    }
}

// files of one call staged at their bound offsets -> packed back to back (the host entry point copies them out in one piece)
struct JpegPackChunk { int64_t src[JPEG_ENC_CHUNK], dst[JPEG_ENC_CHUNK], len[JPEG_ENC_CHUNK]; };
__global__ void __launch_bounds__(256)
jpeg_enc_pack_kernel(const __grid_constant__ JpegPackChunk ch, const uint8_t* __restrict__ src, uint8_t* __restrict__ dst) {
    const int f = blockIdx.y;
    for (int64_t j = blockIdx.x * 256 + threadIdx.x; j < ch.len[f]; j += (int64_t)gridDim.x * 256) dst[ch.dst[f] + j] = src[ch.src[f] + j];
}

}  // namespace yf
