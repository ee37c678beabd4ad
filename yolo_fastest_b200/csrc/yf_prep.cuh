// Pre-processing of Detect_YOLO.__pre_process (reference src/detect.py:107-129) on the GPU: BGR uint8 frames as cv2.imread returns them
// -> cv2.cvtColor(BGR2GRAY) -> cv2.resize(INTER_LINEAR) to the network input size -> uint8 gray planes, which the stem kernel then
// normalises ((x - 128) / 255, detect.py:124) while it loads them. Everything here is the integer arithmetic OpenCV 4.x uses for
// 8-bit images (modules/imgproc color_rgb: 15-bit gray coefficients; resize.cpp: 11-bit interpolation coefficients, HResizeLinear /
// VResizeLinear fixed-point casts), so the result is bit-identical to the host path: oracle/preprocess_oracle.py restates it and is
// pinned against cv2 itself.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace yf {

// one entry per output column / row: the two source indices and the two 11-bit coefficients
struct PrepTap { int s0, s1, c0, c1; };

// resize.cpp (cv::resize, INTER_LINEAR, 8-bit): fx = (float)((dx + 0.5) * scale - 0.5); sx = floor(fx); fx -= sx;
// columns clamp the index AND drop the fraction at both borders, rows keep the fraction and clip the two source rows
inline void prep_taps(int dst_n, int src_n, bool is_row, PrepTap* out) {
    const double inv_scale = (double)dst_n / src_n, scale = 1.0 / inv_scale;
    for (int d = 0; d < dst_n; ++d) {
        float f = (float)((d + 0.5) * scale - 0.5);
        int s = (int)floorf(f);
        f -= (float)s;
        int s0, s1;
        if (is_row) {
            s0 = s < 0 ? 0 : (s > src_n - 1 ? src_n - 1 : s);
            s1 = s + 1 < 0 ? 0 : (s + 1 > src_n - 1 ? src_n - 1 : s + 1);
        } else {
            if (s < 0) { f = 0.f; s = 0; }
            if (s >= src_n - 1) { f = 0.f; s = src_n - 1; }
            s0 = s; s1 = s + 1 > src_n - 1 ? src_n - 1 : s + 1;
        }
        const int c0 = (int)lrintf((1.f - f) * 2048.f), c1 = (int)lrintf(f * 2048.f);           // cvRound: half to even
        if (c1 == 0) s1 = s0;                           // the second tap does not contribute: never fetch it
        out[d] = {s0, s1, c0, c1};
    }
}

// The three integer steps every pre-processing kernel shares (one definition each):
__host__ __device__ __forceinline__ int prep_y(int b, int g, int r) {       // BGR -> Y, 15-bit coefficients (B 3735, G 19235, R 9798)
    return (b * 3735 + g * 19235 + r * 9798 + (1 << 14)) >> 15;
}
__device__ __forceinline__ int prep_hlin(int a, int b, const PrepTap& t) { return a * t.c0 + b * t.c1; }    // HResizeLinear: 11-bit scaled
__device__ __forceinline__ int prep_vlin(int h0, int h1, const PrepTap& t) {                                  // VResizeLinear fixed-point cast
    return (((t.c0 * (h0 >> 4)) >> 16) + ((t.c1 * (h1 >> 4)) >> 16) + 2) >> 2;
}

__device__ __forceinline__ int prep_gray(const uint8_t* __restrict__ p) { return prep_y(__ldg(p), __ldg(p + 1), __ldg(p + 2)); }

// thread = 4 consecutive output pixels of one row (one 32-bit store); grid-stride over [B][H][W / 4]
__global__ void __launch_bounds__(256)
prep_bgr_kernel(const uint8_t* __restrict__ bgr, uint8_t* __restrict__ gray, const PrepTap* __restrict__ xt, const PrepTap* __restrict__ yt,
                int B, int Ho, int Wo, int H, int W) {
    const int W4 = W >> 2;
    const long long total = (long long)B * H * W4;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int q = (int)(i % W4);
        const long long rest = i / W4;
        const int y = (int)(rest % H), b = (int)(rest / H);
        const PrepTap ty = yt[y];
        const uint8_t* r0 = bgr + ((size_t)b * Ho + ty.s0) * (size_t)Wo * 3;
        const uint8_t* r1 = bgr + ((size_t)b * Ho + ty.s1) * (size_t)Wo * 3;
        uint32_t packed = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const PrepTap tx = xt[q * 4 + k];
            const int h0 = prep_hlin(prep_gray(r0 + tx.s0 * 3), prep_gray(r0 + tx.s1 * 3), tx);
            const int h1 = prep_hlin(prep_gray(r1 + tx.s0 * 3), prep_gray(r1 + tx.s1 * 3), tx);
            const int v = prep_vlin(h0, h1, ty);
            packed |= (uint32_t)(v & 255) << (8 * k);
        }
        *reinterpret_cast<uint32_t*>(gray + ((size_t)b * H + y) * W + q * 4) = packed;
    }
}

// Row-staged form (frame width a multiple of 4, 4-byte aligned frames): a block owns PREP_R output rows at a time. Their source rows
// are read ONCE, as coalesced 32-bit words with every load of the group in flight together, converted to gray and kept in shared
// memory; the threads then interpolate 4 consecutive output pixels each from those bytes. Every frame byte is fetched from HBM exactly
// once for identity and integer down-scales. blockDim.x = k * (Wo / 4) >= W / 4; dynamic shared memory = 2 * PREP_R * Wo bytes.
constexpr int PREP_R = 8;
__device__ __forceinline__ uint32_t prep_gray4(uint32_t w0, uint32_t w1, uint32_t w2) {      // 4 BGR pixels (12 bytes) -> 4 gray bytes
    auto byte = [](uint32_t w, int k) { return (int)__byte_perm(w, 0, 0x4440 + k); };
    auto y = [](int b, int g, int r) { return (uint32_t)prep_y(b, g, r); };
    return y(byte(w0, 0), byte(w0, 1), byte(w0, 2)) | (y(byte(w0, 3), byte(w1, 0), byte(w1, 1)) << 8) |
           (y(byte(w1, 2), byte(w1, 3), byte(w2, 0)) << 16) | (y(byte(w2, 1), byte(w2, 2), byte(w2, 3)) << 24);
}

__global__ void __launch_bounds__(1024)
prep_bgr_rows_kernel(const uint8_t* __restrict__ bgr, uint8_t* __restrict__ gray, const PrepTap* __restrict__ xt, const PrepTap* __restrict__ yt,
                     int B, int Ho, int Wo, int H, int W) {
    extern __shared__ uint32_t prep_sm[];               // [2 * PREP_R rows][Wo / 4] words of gray bytes
    __shared__ int srow[2 * PREP_R];                    // source row staged in each slot, -1 = not needed
    __shared__ PrepTap tys[PREP_R];
    const int W4 = W >> 2, Wo4 = Wo >> 2, tid = (int)threadIdx.x;
    const int sr = tid / Wo4, sg = tid - sr * Wo4, sk = (int)blockDim.x / Wo4;          // staging role: rows sr, sr + sk, ..; word group sg
    const int orow = tid / W4, oq = tid - orow * W4, ok = (int)blockDim.x / W4;         // output role: rows orow, orow + ok, ..; pixels 4 oq ..
    PrepTap tx[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) tx[k] = xt[min(oq, W4 - 1) * 4 + k];
    const int groups = (H + PREP_R - 1) / PREP_R;       // row groups per image
    for (long long it = blockIdx.x; it < (long long)B * groups; it += gridDim.x) {
        const int b = (int)(it / groups), y0 = (int)(it - (long long)b * groups) * PREP_R;
        if (tid < PREP_R) {
            const int yy = y0 + tid;
            PrepTap t = yt[min(yy, H - 1)];
            tys[tid] = t;
            srow[2 * tid] = yy < H ? t.s0 : -1;
            srow[2 * tid + 1] = (yy < H && t.s1 != t.s0) ? t.s1 : -1;
        }
        __syncthreads();
        if (sr < sk) {
            const uint8_t* img = bgr + (size_t)b * Ho * (size_t)Wo * 3;
#pragma unroll 4
            for (int ri = sr; ri < 2 * PREP_R; ri += sk) {
                const int r = srow[ri];
                if (r >= 0) {
                    const uint32_t* src = reinterpret_cast<const uint32_t*>(img + (size_t)r * Wo * 3) + 3 * sg;
                    prep_sm[ri * Wo4 + sg] = prep_gray4(__ldg(src), __ldg(src + 1), __ldg(src + 2));
                }
            }
        }
        __syncthreads();
        if (orow < ok) {
            for (int ro = orow; ro < PREP_R && y0 + ro < H; ro += ok) {
                const PrepTap ty = tys[ro];
                const uint8_t* g0 = reinterpret_cast<const uint8_t*>(prep_sm + (2 * ro) * Wo4);
                const uint8_t* g1 = ty.s1 == ty.s0 ? g0 : reinterpret_cast<const uint8_t*>(prep_sm + (2 * ro + 1) * Wo4);
                uint32_t packed = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int h0 = prep_hlin(g0[tx[k].s0], g0[tx[k].s1], tx[k]);
                    const int h1 = prep_hlin(g1[tx[k].s0], g1[tx[k].s1], tx[k]);
                    const int v = prep_vlin(h0, h1, ty);
                    packed |= (uint32_t)(v & 255) << (8 * k);
                }
                *reinterpret_cast<uint32_t*>(gray + ((size_t)b * H + y0 + ro) * W + oq * 4) = packed;
            }
        }
        __syncthreads();
    }
}

// ---- frames of any size in one launch (yf_preprocess_frames / yf_detect_host_frames) ------------------------------------------------
// Frame b of a launch is [Ho, Wo, 3] BGR bytes at frames + off, rows contiguous. Its taps are computed in the kernel instead of read
// from a host table, so a batch may mix sizes without an upload or a synchronisation. The descriptors travel by value in the kernel
// parameters, PREP_CHUNK of them per launch (8 KB), so no device-side descriptor buffer can race with an earlier launch.
struct PrepFrame { int64_t off; int32_t Ho, Wo; };
constexpr int PREP_CHUNK = 512;
struct PrepFrames { PrepFrame f[PREP_CHUNK]; };
constexpr int PREP_SMEM_CAP = 200 * 1024;               // dynamic shared memory a launch may opt in to (frames up to 12800 / 4266 px wide)

// prep_taps, computed on the device operation for operation: every step is an explicitly rounded intrinsic, so nvcc can contract
// nothing into an FMA and the coefficients equal the host table's bit for bit.
__device__ __forceinline__ double prep_scale(int dst_n, int src_n) { return __ddiv_rn(1.0, __ddiv_rn((double)dst_n, (double)src_n)); }
__device__ __forceinline__ PrepTap prep_tap(int d, int src_n, double scale, bool is_row) {
    float f = __double2float_rn(__dsub_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), 0.5));
    int s = (int)floorf(f);
    f = __fsub_rn(f, (float)s);
    int s0, s1;
    if (is_row) {
        s0 = s < 0 ? 0 : (s > src_n - 1 ? src_n - 1 : s);
        s1 = s + 1 < 0 ? 0 : (s + 1 > src_n - 1 ? src_n - 1 : s + 1);
    } else {
        if (s < 0) { f = 0.f; s = 0; }
        if (s >= src_n - 1) { f = 0.f; s = src_n - 1; }
        s0 = s; s1 = s + 1 > src_n - 1 ? src_n - 1 : s + 1;
    }
    const int c0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f)), c1 = __float2int_rn(__fmul_rn(f, 2048.f));
    if (c1 == 0) s1 = s0;
    return {s0, s1, c0, c1};
}

// A frame is staged in shared memory when its rows can be read as 32-bit words (width a multiple of 4, so the 3 * Wo byte pitch is
// too, and a 4-byte aligned base) and its 2 * PREP_R source rows fit the launch's dynamic shared memory; otherwise it is read with
// byte loads from global memory. The host sizes the shared memory with the same rule.
__host__ __device__ __forceinline__ int prep_stage_bytes(int Wo, int ch) { return 2 * PREP_R * Wo * ch; }
__host__ __device__ __forceinline__ bool prep_stageable(const uint8_t* frames, const PrepFrame& f, int ch, int smem_bytes) {
    return f.Wo % 4 == 0 && (((uintptr_t)frames + (uintptr_t)f.off) & 3) == 0 && prep_stage_bytes(f.Wo, ch) <= smem_bytes;
}

// 4 consecutive output pixels of one output row, every plane: px(r, s, c) = byte c of source pixel s in source row r (0: ty.s0, 1: ty.s1)
template <int CH, class Px>
__device__ __forceinline__ void prep_store4(const Px& px, const PrepTap& ty, const PrepTap (&tx)[4], uint8_t* dst, size_t plane) {
#pragma unroll
    for (int c = 0; c < CH; ++c) {
        const int sc = CH == 3 ? 2 - c : 0;             // planes R, G, B out of interleaved B, G, R (detect.py:121, [:, :, ::-1])
        uint32_t packed = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int h0 = prep_hlin(px(0, tx[k].s0, sc), px(0, tx[k].s1, sc), tx[k]);
            const int h1 = prep_hlin(px(1, tx[k].s0, sc), px(1, tx[k].s1, sc), tx[k]);
            packed |= (uint32_t)(prep_vlin(h0, h1, ty) & 255) << (8 * k);
        }
        *reinterpret_cast<uint32_t*>(dst + c * plane) = packed;
    }
}

// this thread's pixel groups of one output row: group oq with the cached column taps when the row fits the block (one group per
// thread), else groups oq, oq + oqs, .. with their taps computed as they come
template <int CH, class Px>
__device__ __forceinline__ void prep_row(const Px& px, const PrepTap& ty, const PrepTap (&tx)[4], bool ofit, int oq, int oqs, int W4,
                                         int Wo, double sx, uint8_t* drow, size_t plane) {
    if (ofit) {
        prep_store4<CH>(px, ty, tx, drow + oq * 4, plane);
        return;
    }
    for (int q = oq; q < W4; q += oqs) {
        PrepTap t[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) t[k] = prep_tap(q * 4 + k, Wo, sx, false);
        prep_store4<CH>(px, ty, t, drow + q * 4, plane);
    }
}

// CH = 1: out [nf, H, W] gray (cvtColor BGR2GRAY, then resize). CH = 3: out [nf, 3, H, W] R, G, B planes (resize of each channel,
// then the channel flip) — the same 11-bit arithmetic once per channel, which is what cv2.resize does with a 3-channel uint8 image.
// Grid-stride over (frame, group of PREP_R output rows) as prep_bgr_rows_kernel; a staged frame's source rows are read once with 32-bit
// loads (3 words = 4 pixels per unit) and kept in shared memory as gray bytes (CH = 1) or BGR bytes (CH = 3).
constexpr int PREP_NT = 512;                            // threads per block of prep_frames_kernel
template <int CH>
__global__ void __launch_bounds__(PREP_NT, CH == 1 ? 2 : 1)
prep_frames_kernel(const uint8_t* __restrict__ frames, const __grid_constant__ PrepFrames fr, int nf, uint8_t* __restrict__ out,
                   int H, int W, int smem_bytes) {
    extern __shared__ uint32_t prep_sm[];               // [2 * PREP_R slots][Wo / 4 units] x (CH == 1 ? 1 : 3) words
    __shared__ int srow[2 * PREP_R];                    // source row staged in each slot, -1 = not needed
    __shared__ PrepTap tys[PREP_R];
    const int W4 = W >> 2, tid = (int)threadIdx.x, nt = (int)blockDim.x;
    const bool ofit = W4 <= nt;                         // output role: rows orow, orow + ok, ..; pixel groups oq, oq + oqs, ..
    const int orow = ofit ? tid / W4 : 0, oq = ofit ? tid - orow * W4 : tid, ok = ofit ? nt / W4 : 1, oqs = ofit ? W4 : nt;
    const size_t plane = (size_t)H * W;
    int cur_Wo = 0, cur_Ho = 0, G = 0, sr = 0, sg = 0, sk = 0;       // staging role (sfit): rows sr, sr + sk, ..; unit sg
    bool sfit = false;
    double sx = 0.0, sy = 0.0;
    PrepTap tx[4];
    const int groups = (H + PREP_R - 1) / PREP_R;
    for (long long it = blockIdx.x; it < (long long)nf * groups; it += gridDim.x) {
        const int b = (int)(it / groups), y0 = (int)(it - (long long)b * groups) * PREP_R;
        const PrepFrame f = fr.f[b];
        if (f.Wo != cur_Wo) {                           // column taps and staging role of this width (kept while the width repeats)
            cur_Wo = f.Wo;
            sx = prep_scale(W, f.Wo);
#pragma unroll
            for (int k = 0; k < 4; ++k) tx[k] = prep_tap(min(oq, W4 - 1) * 4 + k, f.Wo, sx, false);
            G = f.Wo >> 2;
            sfit = G > 0 && G <= nt;
            if (sfit) { sr = tid / G; sg = tid - sr * G; sk = nt / G; }
        }
        if (tid < PREP_R) {
            const int yy = y0 + tid;
            if (f.Ho != cur_Ho) { cur_Ho = f.Ho; sy = prep_scale(H, f.Ho); }
            const PrepTap t = prep_tap(min(yy, H - 1), f.Ho, sy, true);
            tys[tid] = t;
            srow[2 * tid] = yy < H ? t.s0 : -1;
            srow[2 * tid + 1] = (yy < H && t.s1 != t.s0) ? t.s1 : -1;
        }
        __syncthreads();
        const uint8_t* img = frames + f.off;
        const size_t pitch = (size_t)f.Wo * 3;
        uint8_t* dimg = out + (size_t)b * CH * plane;
        if (prep_stageable(frames, f, CH, smem_bytes)) {
            constexpr int UW = CH == 1 ? 1 : 3;         // staged words per 4-pixel unit
            auto stage = [&](int ri, int g, const uint32_t* src) {
                const uint32_t w0 = __ldg(src + 3 * g), w1 = __ldg(src + 3 * g + 1), w2 = __ldg(src + 3 * g + 2);
                if (CH == 1) {
                    prep_sm[ri * G + g] = prep_gray4(w0, w1, w2);
                } else {
                    uint32_t* d = prep_sm + (ri * G + g) * 3;
                    d[0] = w0; d[1] = w1; d[2] = w2;
                }
            };
            if (sfit) {                                 // a staged row fits the block: one unit per thread and row, loads in flight together
                if (sr < sk) {
#pragma unroll 4
                    for (int ri = sr; ri < 2 * PREP_R; ri += sk) {
                        const int r = srow[ri];
                        if (r >= 0) stage(ri, sg, reinterpret_cast<const uint32_t*>(img + (size_t)r * pitch));
                    }
                }
            } else {
                for (int ri = 0; ri < 2 * PREP_R; ++ri) {
                    const int r = srow[ri];
                    if (r >= 0)
                        for (int g = tid; g < G; g += nt) stage(ri, g, reinterpret_cast<const uint32_t*>(img + (size_t)r * pitch));
                }
            }
            __syncthreads();
            if (orow < ok) {
                for (int ro = orow; ro < PREP_R && y0 + ro < H; ro += ok) {
                    const PrepTap ty = tys[ro];
                    const uint8_t* g0 = reinterpret_cast<const uint8_t*>(prep_sm + (2 * ro) * G * UW);
                    const uint8_t* g1 = ty.s1 == ty.s0 ? g0 : reinterpret_cast<const uint8_t*>(prep_sm + (2 * ro + 1) * G * UW);
                    auto px = [&](int r, int s, int c) { return (int)(r ? g1 : g0)[CH == 1 ? s : 3 * s + c]; };
                    prep_row<CH>(px, ty, tx, ofit, oq, oqs, W4, f.Wo, sx, dimg + (size_t)(y0 + ro) * W, plane);
                }
            }
        } else if (orow < ok) {                         // byte loads from global memory: any width, any alignment
            for (int ro = orow; ro < PREP_R && y0 + ro < H; ro += ok) {
                const PrepTap ty = tys[ro];
                const uint8_t* r0 = img + (size_t)ty.s0 * pitch;
                const uint8_t* r1 = img + (size_t)ty.s1 * pitch;
                auto px = [&](int r, int s, int c) { return CH == 1 ? prep_gray((r ? r1 : r0) + 3 * s) : (int)__ldg((r ? r1 : r0) + 3 * s + c); };
                prep_row<CH>(px, ty, tx, ofit, oq, oqs, W4, f.Wo, sx, dimg + (size_t)(y0 + ro) * W, plane);
            }
        }
        __syncthreads();
    }
}

}  // namespace yf
