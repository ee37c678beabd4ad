// YUV 4:2:0 frames (NV12, I420) on the device: the BGR frame cv2.cvtColor(frame, COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420) returns,
// and the network input detect.py:107-122 computes from that BGR frame, without writing the BGR frame to memory. A frame is three
// planes described by byte offsets from one base pointer (yf_yuv420, include/yf.h): chroma sample k of chroma row r is at
// u_off + r * c_pitch + k * c_step (NV12: c_step 2, v_off = u_off + 1; I420: c_step 1, separate planes). Pixel (r, c) uses chroma
// sample (r / 2, c / 2): cv2 does not interpolate chroma for these codes. The kernels never branch on the format.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/yf.h"
#include "yf_prep.cuh"

namespace yf {

// cv2 4.x color_yuv (YUV420 -> BGR, 8-bit): BT.601 limited range in 20-bit fixed point; every intermediate fits in int32.
// -> B | G << 8 | R << 16, the byte order of a packed BGR pixel.
__host__ __device__ __forceinline__ uint32_t yuv_sat(int x) { return (uint32_t)(x < 0 ? 0 : (x > 255 ? 255 : x)); }
__host__ __device__ __forceinline__ uint32_t yuv_bgr(int Y, int U, int V) {
    const int y = (Y > 16 ? Y - 16 : 0) * 1220542 + (1 << 19), u = U - 128, v = V - 128;
    const uint32_t r = yuv_sat((y + 1673527 * v) >> 20);
    const uint32_t g = yuv_sat((y - 852492 * v - 409993 * u) >> 20);
    const uint32_t b = yuv_sat((y + 2116026 * u) >> 20);
    return b | (g << 8) | (r << 16);
}
__device__ __forceinline__ int yuv_gray(uint32_t p) { return prep_y((int)(p & 255), (int)((p >> 8) & 255), (int)(p >> 16)); }

// 4 consecutive packed pixels -> the 12 BGR bytes as 3 little-endian words
__device__ __forceinline__ void yuv_words(uint32_t p0, uint32_t p1, uint32_t p2, uint32_t p3, uint32_t& w0, uint32_t& w1, uint32_t& w2) {
    w0 = p0 | (p1 << 24);
    w1 = (p1 >> 8) | (p2 << 16);
    w2 = (p2 >> 16) | (p3 << 8);
}

// Descriptors travel by value in the kernel parameters (12 KB + 2 KB), YUV_CHUNK of them per launch, as in prep_frames_kernel.
constexpr int YUV_CHUNK = 256;
struct YuvFrames { yf_yuv420 f[YUV_CHUNK]; };
struct YuvBgrFrames { yf_yuv420 f[YUV_CHUNK]; int64_t dst[YUV_CHUNK]; };

// ---- conversion: frame blockIdx.y of the chunk -> [h, w, 3] BGR bytes at frames + dst, contiguous rows ------------------------------
// thread = 4 columns x 2 rows (the pixels of two chroma samples); 3 word stores per row when the output rows are 4-byte aligned
constexpr int YUV_NT = 256;
__global__ void __launch_bounds__(YUV_NT)
yuv_bgr_kernel(const uint8_t* __restrict__ base, const __grid_constant__ YuvBgrFrames ch, uint8_t* __restrict__ frames) {
    const yf_yuv420 f = ch.f[blockIdx.y];
    uint8_t* dimg = frames + ch.dst[blockIdx.y];
    const int q4 = (f.w + 3) >> 2;
    const long long units = (long long)(f.h >> 1) * q4;
    const bool wstore = (f.w & 3) == 0 && ((uintptr_t)dimg & 3) == 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < units; i += (long long)gridDim.x * blockDim.x) {
        const int cr = (int)(i / q4), c0 = 4 * (int)(i - (long long)cr * q4);
        const int n = min(4, f.w - c0);                 // 4, or 2 at the end of a row of width 2 mod 4
        const uint8_t* ur = base + f.u_off + (size_t)cr * f.c_pitch + (size_t)(c0 >> 1) * f.c_step;
        const uint8_t* vr = base + f.v_off + (size_t)cr * f.c_pitch + (size_t)(c0 >> 1) * f.c_step;
        const int U0 = __ldg(ur), V0 = __ldg(vr);
        const int U1 = n == 4 ? __ldg(ur + f.c_step) : 0, V1 = n == 4 ? __ldg(vr + f.c_step) : 0;
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int row = 2 * cr + r;
            const uint8_t* yr = base + f.y_off + (size_t)row * f.y_pitch + c0;
            uint8_t* d = dimg + ((size_t)row * f.w + c0) * 3;
            const uint32_t p0 = yuv_bgr(__ldg(yr), U0, V0), p1 = yuv_bgr(__ldg(yr + 1), U0, V0);
            if (n == 4) {
                const uint32_t p2 = yuv_bgr(__ldg(yr + 2), U1, V1), p3 = yuv_bgr(__ldg(yr + 3), U1, V1);
                if (wstore) {
                    uint32_t w0, w1, w2;
                    yuv_words(p0, p1, p2, p3, w0, w1, w2);
                    uint32_t* dw = reinterpret_cast<uint32_t*>(d);
                    dw[0] = w0; dw[1] = w1; dw[2] = w2;
                } else {
                    const uint32_t p[4] = {p0, p1, p2, p3};
#pragma unroll
                    for (int k = 0; k < 4; ++k) { d[3 * k] = (uint8_t)p[k]; d[3 * k + 1] = (uint8_t)(p[k] >> 8); d[3 * k + 2] = (uint8_t)(p[k] >> 16); }
                }
            } else {
                d[0] = (uint8_t)p0; d[1] = (uint8_t)(p0 >> 8); d[2] = (uint8_t)(p0 >> 16);
                d[3] = (uint8_t)p1; d[4] = (uint8_t)(p1 >> 8); d[5] = (uint8_t)(p1 >> 16);
            }
        }
    }
}

// ---- fused pre-processing: YUV planes -> gray [nf, H, W] or R, G, B planes [nf, 3, H, W], no BGR frame in memory ------------------
// A frame is staged when its luma rows and both chroma rows can be read as aligned 32-bit words: width a multiple of 4, luma rows
// 4-byte aligned, chroma pitch a multiple of 4 and the two chroma samples of every 4-pixel unit inside one aligned word (c_step 1 with
// even plane starts, c_step 2 with plane starts at 0 or 1 mod 4: the U and V planes of NV12), and its 2 * PREP_R source rows fit the
// launch's dynamic shared memory. Any other frame is read with byte loads. The host sizes the shared memory with the same rule.
__host__ __device__ __forceinline__ bool yuv_pairs_in_words(uintptr_t plane, int c_pitch, int c_step) {
    return (c_pitch & 3) == 0 && (c_step == 1 ? (plane & 1) == 0 : c_step == 2 && (plane & 3) <= 1);
}
__host__ __device__ __forceinline__ bool yuv_stageable(const uint8_t* base, const yf_yuv420& f, int ch, int smem_bytes) {
    const uintptr_t a = (uintptr_t)base;
    return f.w % 4 == 0 && ((a + (uintptr_t)f.y_off) & 3) == 0 && (f.y_pitch & 3) == 0 &&
           yuv_pairs_in_words(a + (uintptr_t)f.u_off, f.c_pitch, f.c_step) && yuv_pairs_in_words(a + (uintptr_t)f.v_off, f.c_pitch, f.c_step) &&
           prep_stage_bytes(f.w, ch) <= smem_bytes;
}

// the same grid-stride over (frame, group of PREP_R output rows), taps and output role as prep_frames_kernel; only the source differs
template <int CH>
__global__ void __launch_bounds__(PREP_NT, CH == 1 ? 2 : 1)
prep_yuv_kernel(const uint8_t* __restrict__ base, const __grid_constant__ YuvFrames fr, int nf, uint8_t* __restrict__ out,
                int H, int W, int smem_bytes) {
    extern __shared__ uint32_t prep_sm[];               // [2 * PREP_R slots][w / 4 units] x (CH == 1 ? 1 : 3) words
    __shared__ int srow[2 * PREP_R];                    // source row staged in each slot, -1 = not needed
    __shared__ PrepTap tys[PREP_R];
    const int W4 = W >> 2, tid = (int)threadIdx.x, nt = (int)blockDim.x;
    const bool ofit = W4 <= nt;
    const int orow = ofit ? tid / W4 : 0, oq = ofit ? tid - orow * W4 : tid, ok = ofit ? nt / W4 : 1, oqs = ofit ? W4 : nt;
    const size_t plane = (size_t)H * W;
    int cur_w = 0, cur_h = 0, G = 0, sr = 0, sg = 0, sk = 0;
    bool sfit = false;
    double sx = 0.0, sy = 0.0;
    PrepTap tx[4];
    const int groups = (H + PREP_R - 1) / PREP_R;
    for (long long it = blockIdx.x; it < (long long)nf * groups; it += gridDim.x) {
        const int b = (int)(it / groups), y0 = (int)(it - (long long)b * groups) * PREP_R;
        const yf_yuv420& f = fr.f[b];           // read from the parameter bank, not held in registers
        if (f.w != cur_w) {
            cur_w = f.w;
            sx = prep_scale(W, f.w);
#pragma unroll
            for (int k = 0; k < 4; ++k) tx[k] = prep_tap(min(oq, W4 - 1) * 4 + k, f.w, sx, false);
            G = f.w >> 2;
            sfit = G > 0 && G <= nt;
            if (sfit) { sr = tid / G; sg = tid - sr * G; sk = nt / G; }
        }
        if (tid < PREP_R) {
            const int yy = y0 + tid;
            if (f.h != cur_h) { cur_h = f.h; sy = prep_scale(H, f.h); }
            const PrepTap t = prep_tap(min(yy, H - 1), f.h, sy, true);
            tys[tid] = t;
            srow[2 * tid] = yy < H ? t.s0 : -1;
            srow[2 * tid + 1] = (yy < H && t.s1 != t.s0) ? t.s1 : -1;
        }
        __syncthreads();
        const uint8_t* yp = base + f.y_off;
        const uint8_t* up = base + f.u_off;
        const uint8_t* vp = base + f.v_off;
        uint8_t* dimg = out + (size_t)b * CH * plane;
        if (yuv_stageable(base, f, CH, smem_bytes)) {
            constexpr int UW = CH == 1 ? 1 : 3;
            auto stage = [&](int ri, int g, int r) {    // unit g (pixels 4g .. 4g + 3) of source row r -> gray or BGR bytes
                const uint32_t y4 = __ldg(reinterpret_cast<const uint32_t*>(yp + (size_t)r * f.y_pitch) + g);
                const size_t co = (size_t)(r >> 1) * f.c_pitch + (size_t)(2 * g) * f.c_step;
                const uintptr_t ua = (uintptr_t)(up + co), va = (uintptr_t)(vp + co);
                const uint32_t uw = __ldg(reinterpret_cast<const uint32_t*>(ua & ~(uintptr_t)3));
                const uint32_t vw = __ldg(reinterpret_cast<const uint32_t*>(va & ~(uintptr_t)3));
                const int us = 8 * (int)(ua & 3), vs = 8 * (int)(va & 3), ss = 8 * f.c_step;
                const int U0 = (uw >> us) & 255, U1 = (uw >> (us + ss)) & 255, V0 = (vw >> vs) & 255, V1 = (vw >> (vs + ss)) & 255;
                const uint32_t p0 = yuv_bgr(y4 & 255, U0, V0), p1 = yuv_bgr((y4 >> 8) & 255, U0, V0);
                const uint32_t p2 = yuv_bgr((y4 >> 16) & 255, U1, V1), p3 = yuv_bgr(y4 >> 24, U1, V1);
                if (CH == 1) {
                    prep_sm[ri * G + g] = (uint32_t)yuv_gray(p0) | ((uint32_t)yuv_gray(p1) << 8) | ((uint32_t)yuv_gray(p2) << 16) |
                                          ((uint32_t)yuv_gray(p3) << 24);
                } else {
                    uint32_t* d = prep_sm + (ri * G + g) * 3;
                    yuv_words(p0, p1, p2, p3, d[0], d[1], d[2]);
                }
            };
            if (sfit) {
                if (sr < sk) {
#pragma unroll 4
                    for (int ri = sr; ri < 2 * PREP_R; ri += sk) {
                        const int r = srow[ri];
                        if (r >= 0) stage(ri, sg, r);
                    }
                }
            } else {
                for (int ri = 0; ri < 2 * PREP_R; ++ri) {
                    const int r = srow[ri];
                    if (r >= 0)
                        for (int g = tid; g < G; g += nt) stage(ri, g, r);
                }
            }
            __syncthreads();
            if (orow < ok) {
                for (int ro = orow; ro < PREP_R && y0 + ro < H; ro += ok) {
                    const PrepTap ty = tys[ro];
                    const uint8_t* g0 = reinterpret_cast<const uint8_t*>(prep_sm + (2 * ro) * G * UW);
                    const uint8_t* g1 = ty.s1 == ty.s0 ? g0 : reinterpret_cast<const uint8_t*>(prep_sm + (2 * ro + 1) * G * UW);
                    auto px = [&](int r, int s, int c) { return (int)(r ? g1 : g0)[CH == 1 ? s : 3 * s + c]; };
                    prep_row<CH>(px, ty, tx, ofit, oq, oqs, W4, f.w, sx, dimg + (size_t)(y0 + ro) * W, plane);
                }
            }
        } else if (orow < ok) {                         // byte loads from global memory: any pitch, step and alignment
            for (int ro = orow; ro < PREP_R && y0 + ro < H; ro += ok) {
                const PrepTap ty = tys[ro];
                const uint8_t* y0r = yp + (size_t)ty.s0 * f.y_pitch;
                const uint8_t* y1r = yp + (size_t)ty.s1 * f.y_pitch;
                const size_t c0 = (size_t)(ty.s0 >> 1) * f.c_pitch, c1 = (size_t)(ty.s1 >> 1) * f.c_pitch;
                auto px = [&](int r, int s, int c) {
                    const size_t co = (r ? c1 : c0) + (size_t)(s >> 1) * f.c_step;
                    const uint32_t p = yuv_bgr(__ldg((r ? y1r : y0r) + s), __ldg(up + co), __ldg(vp + co));
                    return CH == 1 ? yuv_gray(p) : (int)((p >> (8 * c)) & 255);
                };
                prep_row<CH>(px, ty, tx, ofit, oq, oqs, W4, f.w, sx, dimg + (size_t)(y0 + ro) * W, plane);
            }
        }
        __syncthreads();
    }
}

}  // namespace yf
