// yf_tcpw_tma.cuh — the depthwise 5x5 -> wide 1x1 pairs of the neck and the composed heads (yf_tcpw.cuh) with the input fed by
// tensor-tile TMA. Same arithmetic, same packed weights, same MMA sequence as dwpw_tc_kernel, so the two are bit-identical.
//
// What changes against dwpw_tc_kernel:
//   - the halo rectangle of a 16-channel chunk arrives as ONE TMA box {TW + 8, TH + 4, MC, 1} starting at the aligned column ox0 - 4
//     (yf_tma.cuh: the innermost start must be a multiple of 16 bytes), into a ring of NST stages with full / free mbarriers. A producer
//     warp keeps the ring filled across tile boundaries; the TMA zero fill is the convolution's padding. No per-element bounds checks,
//     no cp.async, and no block-wide barrier per chunk: the workers wait on the stage's full barrier and arrive on its free barrier.
//   - the depthwise runs on pixel PAIRS with fma.rn.f32x2 (FFMA2, per-lane rounding of fmaf): a thread owns one channel and a strip of
//     2 columns x RH rows; each 6-float window row (3 LDS.64) feeds up to 5 output rows.
//   - the epilogue of tile t runs after the depthwise of tile t + 1's first chunk, so that chunk's operand is ready when the last MMA of
//     tile t completes. Where two accumulators fit into TMEM (the heads, N = 32) the next tile's MMAs do not wait for the read-out.
#pragma once
#include "yf_tcpw.cuh"
#include "yf_tma.cuh"

namespace yf {

// rows per depthwise item: the tallest strip that still gives every worker thread an item (fewer window reloads per output row)
constexpr int dwpw_tma_rh(int TH, int TW, int MC, int NTW) {
    for (int rh = 8; rh > 1; rh >>= 1)
        if (TH % rh == 0 && MC * (TH / rh) * (TW / 2) >= NTW) return rh;
    return 1;
}

template <class B>
struct DwPwTmaCfg : B {
    using G = typename B::G;
    static constexpr int MC = B::MC, NTW = B::NTW, NWB = B::NWB, CB = B::CB, DA1 = B::DA1, MT3 = B::MT3, NP = B::NP;
    static constexpr int NT = NTW + 64;                                   // workers + the tensor-core warp + the TMA producer warp
    static constexpr int BW = G::TW + 8, BH = G::IH;                      // box columns from ox0 - 4, rows from oy0 - 2
    static constexpr int BOX = MC * BH * BW;                              // floats of one ring stage [MC][BH][BW]
    static constexpr int RH = dwpw_tma_rh(G::TH, G::TW, MC, NTW);
    static constexpr int ACOLS = pow2_ge(MT3 * NP);                       // TMEM columns of one accumulator set
    static constexpr int NACC = 2 * ACOLS <= 512 ? 2 : 1;
    static constexpr int TCOLS = NACC * ACOLS;
    static constexpr int FIXED = 4 * DA1 + NWB * CB;
    static constexpr int NST = (FIXED + 3 * BOX) * 4 + 1024 <= 227 * 1024 ? 3 : 2;
    static constexpr int SMEM_BYTES = (FIXED + NST * BOX) * 4 + 1024;
    static_assert(G::KS == 5 && G::S == 1 && G::P == 2, "5x5 stride 1: the box starts 2 columns left of the halo");
    static_assert(G::TW % 4 == 0 && BW <= 256 && BH <= 256 && MC <= 256, "TMA box dimensions");
    static_assert((BOX * 4) % 128 == 0 && (CB * 4) % 128 == 0, "ring stages stay 128-byte aligned");
    static_assert(SMEM_BYTES <= 227 * 1024, "two ring stages do not fit shared memory");
    static_assert(BOX * 4 >= 4096, "over-read guard behind the operand regions");
    static_assert(G::TH % RH == 0, "row strips");
};

// depthwise 5x5 s1 + bias + ReLU of one chunk from its TMA box [MC][BH][BW] into the A-operand layout of the 1x1 MMA (hi and lo).
// Item = (channel m, strip of output columns 2g, 2g + 1, rows seg * RH ...). Each output is b, then fmaf(w[dy * 5 + dx], x, .) in dy-major,
// dx order — the order of dwk_stage_split — evaluated two pixels at a time.
template <class C>
__device__ __forceinline__ void dwk_tma_stage(int tid, const float* __restrict__ Xb, const float* __restrict__ Wd, const float* __restrict__ bd,
                                              float* __restrict__ DAhi, float* __restrict__ DAlo) {
    using G = typename C::G;
    constexpr int RH = C::RH, NSTRIP = G::TW / 2, NSEG = G::TH / RH, NITEM = C::MC * NSEG * NSTRIP;
    for (int item = tid; item < NITEM; item += C::NTW) {
        const int g = item % NSTRIP, rest = item / NSTRIP;
        const int seg = rest % NSEG, m = rest / NSEG;
        float w[25];
#pragma unroll
        for (int t = 0; t < 25; ++t) w[t] = Wd[m * 25 + t];
        const float b = bd[m];
        // box column 2 is the halo's column 0; the strip's window is halo columns 2g .. 2g + 5
        const float* e = Xb + m * C::BH * C::BW + (seg * RH) * C::BW + 2 * g + 2;
        float2 win[5][5];                                                  // [row][dx]: the input pair under output pixels (2g + dx, 2g + 1 + dx)
        auto load_row = [&](float2 (&r)[5], const float* p) {
            const float2 a = *reinterpret_cast<const float2*>(p);
            const float2 c = *reinterpret_cast<const float2*>(p + 2);
            const float2 d = *reinterpret_cast<const float2*>(p + 4);
            r[0] = a; r[1] = make_float2(a.y, c.x); r[2] = c; r[3] = make_float2(c.y, d.x); r[4] = d;
        };
#pragma unroll
        for (int dd = 0; dd < 4; ++dd) load_row(win[dd + 1], e + dd * C::BW);
#pragma unroll
        for (int oy = 0; oy < RH; ++oy) {
#pragma unroll
            for (int dd = 0; dd < 4; ++dd)
#pragma unroll
                for (int v = 0; v < 5; ++v) win[dd][v] = win[dd + 1][v];
            load_row(win[4], e + (oy + 4) * C::BW);
            float2 a = make_float2(b, b);
#pragma unroll
            for (int dy = 0; dy < 5; ++dy)
#pragma unroll
                for (int dx = 0; dx < 5; ++dx) a = __ffma2_rn(make_float2(w[dy * 5 + dx], w[dy * 5 + dx]), win[dy][dx], a);
            const float v0 = fmaxf(a.x, 0.f), v1 = fmaxf(a.y, 0.f);
            const float h0 = tf32_hi(v0), h1 = tf32_hi(v1);
            const int o = a_idx((seg * RH + oy) * G::TW + 2 * g, m, C::KB3);     // the pair stays inside one 8-pixel run
            *reinterpret_cast<float2*>(DAhi + o) = make_float2(h0, h1);
            *reinterpret_cast<float2*>(DAlo + o) = make_float2(v0 - h0, v1 - h1);
        }
    }
}

template <class C>
__global__ void __launch_bounds__(C::NT, 1)
dwpw_tma_kernel(const __grid_constant__ CUtensorMap xmap, float* __restrict__ y, const float* __restrict__ wts, int H, int W,
                int tiles_x, int tiles_y, int total_tiles, int nout /* output channels actually stored, <= N (head groups: run time) */) {
    using G = typename C::G;
    constexpr int NWW = C::NWW, NCH = C::NCHUNK, NST = C::NST, NACC = C::NACC;
    extern __shared__ unsigned char smem_raw[];
    float* base = reinterpret_cast<float*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    float* Dbuf = base;                          // [2 buffers][hi | lo][DA1]
    float* Xb = Dbuf + 4 * C::DA1;               // [NST stages][MC][BH][BW]: the TMA boxes
    float* Ws = Xb + NST * C::BOX;               // ring of chunk weight blocks
    __shared__ __align__(8) uint64_t wbar[C::NWB], xfull[NST], xfree[NST], dfull[2], dfree[2], ofull[NACC], ofree[NACC];
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        for (int i = 0; i < C::NWB; ++i) mbar_init(&wbar[i], 1);
        for (int i = 0; i < NST; ++i) { mbar_init(&xfull[i], 1); mbar_init(&xfree[i], NWW); }
        for (int i = 0; i < 2; ++i) { mbar_init(&dfull[i], NWW); mbar_init(&dfree[i], 1); }
        for (int i = 0; i < NACC; ++i) { mbar_init(&ofull[i], 1); mbar_init(&ofree[i], NWW); }
        mbar_fence_init();
    }
    if (warp == NWW) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"((uint32_t)C::TCOLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (warp == NWW + 1) tma_prefetch_desc(&xmap);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    pdl_trigger();
    pdl_wait();
    const uint32_t tmem = tmem_slot;

    const int ntile = total_tiles > (int)blockIdx.x ? (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int S = ntile * NCH;
    const int tpi = tiles_x * tiles_y;
    const uint32_t inv_tx = (65536u + (uint32_t)tiles_x - 1u) / (uint32_t)tiles_x;
    auto origin = [&](int ti, int& b, int& oy0, int& ox0) {
        const int tile = (int)blockIdx.x + ti * (int)gridDim.x;
        b = tile / tpi;
        const int t = tile - b * tpi;
        const int ty = (int)(((uint32_t)t * inv_tx) >> 16);
        oy0 = ty * G::TH; ox0 = (t - ty * tiles_x) * G::TW;
    };

    if (warp == NWW) {
        // ================= tensor-core warp: the MMA sequence of dwpw_tc_kernel, accumulator set ti % NACC =================
        if (S > 0 && elect_one()) {
            constexpr uint32_t IDESC = umma_idesc_tf32(C::NP);
            const uint32_t ws = smem_u32(Ws);
            auto issue_w = [&](int q) {
                const int slot = q % C::NWB;
                mbar_expect_tx(&wbar[slot], C::CB * 4);
                bulk_load(Ws + slot * C::CB, wts + (size_t)(q % NCH) * C::CB, C::CB * 4, &wbar[slot]);
            };
            const uint64_t dd0 = umma_desc(smem_u32(Dbuf), 1024, 512, 1);
            const uint64_t dw0 = umma_desc(ws, 128, (C::MC / 4) * 128, 0);
            issue_w(0);
            if (S > 1) issue_w(1);
            for (int q = 0; q < S; ++q) {
                const int b = q & 1, c = q % NCH, ti = q / NCH, ab = ti % NACC;
                if (c == 0 && ti >= NACC) mbar_wait(&ofree[ab], ((ti / NACC) - 1) & 1);   // this accumulator set has been read out
                mbar_wait(&dfull[b], (q >> 1) & 1);
                mbar_wait(&wbar[q % C::NWB], (q / C::NWB) & 1);
                tc_fence_after();
                const uint64_t wb = dw0 + (uint64_t)(((uint32_t)(q % C::NWB) * C::CB * 4) >> 4);
                const uint64_t db = dd0 + (uint64_t)((uint32_t)(b * 2 * C::DA1 * 4) >> 4);
                const uint32_t acc = tmem + (uint32_t)(ab * C::ACOLS);
#pragma unroll 1
                for (int mt = 0; mt < C::MT3; ++mt) {
                    const uint64_t mo = (uint64_t)(mt * 256);
#pragma unroll
                    for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
                        for (int kb = 0; kb < C::MC / 8; ++kb)
                            umma_tf32(acc + mt * C::NP, db + mo + (uint64_t)(((pass == 2 ? C::DA1 : 0) + kb * C::KB3) * 4 / 16),
                                      wb + (uint64_t)(((pass == 1 ? C::OFF_WL : C::OFF_WH) * 4 + kb * 256) / 16), IDESC,
                                      (c | pass | kb) ? 1u : 0u);
                    }
                }
                umma_commit(&dfree[b]);
                if (c == NCH - 1) umma_commit(&ofull[ab]);
                if (q + 2 < S) {
                    if (q >= 1) mbar_wait(&dfree[(q - 1) & 1], ((q - 1) >> 1) & 1);   // ring slot (q+2)%3 == (q-1)%3 is free
                    issue_w(q + 2);
                }
            }
        }
    } else if (warp == NWW + 1) {
        // ================= TMA producer: the box of every chunk of every tile, NST stages ahead of the workers =================
        if (S > 0 && elect_one()) {
            int q = 0;
            for (int ti = 0; ti < ntile; ++ti) {
                int b, oy0, ox0;
                origin(ti, b, oy0, ox0);
#pragma unroll 1
                for (int c = 0; c < NCH; ++c, ++q) {
                    const int st = q % NST;
                    if (q >= NST) mbar_wait(&xfree[st], ((q / NST) - 1) & 1);   // every worker warp is done with this stage
                    mbar_expect_tx(&xfull[st], C::BOX * 4);
                    tma_load4(Xb + st * C::BOX, &xmap, &xfull[st], ox0 - 4, oy0 - G::P, c * C::MC, b);
                }
            }
        }
    } else {
        // ================= worker warps =================
        const int quarter = warp & 3, wq = warp >> 2;
        const int nwq = (NWW - quarter + 3) >> 2;
        const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
        const size_t plane = (size_t)H * W;
        // ---- epilogue of tile ti: TMEM -> + bias -> HBM (thread = pixel, 16 output channels per unit) --------------------------------
        auto epilogue = [&](int ti) {
            int tb, oy0, ox0;
            origin(ti, tb, oy0, ox0);
            const int ab = ti % NACC;
            mbar_wait(&ofull[ab], (ti / NACC) & 1);
            tc_fence_after();
            for (int u = wq; u < C::MT3 * (C::NP / 16); u += nwq) {
                const int mt = u / (C::NP / 16), c0 = (u - mt * (C::NP / 16)) * 16;
                if (mt * 128 + quarter * 32 >= G::OPIX) break;
                const int pix = mt * 128 + quarter * 32 + lane;
                const int oy = pix / G::TW, ox = pix - oy * G::TW;
                const int gy = oy0 + oy, gx = ox0 + ox;
                float v[16];
                tmem_ld16(tmem + lane_base + (uint32_t)(ab * C::ACOLS) + mt * C::NP + c0, v);
                if (pix < G::OPIX && gy < H && gx < W) {
                    const int nch = C::NRT ? nout : C::N;
                    float* yp = y + ((size_t)tb * nch + c0) * plane + (size_t)gy * W + gx;
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        if (c0 + i < nch) {
                            float r = v[i] + __ldg(wts + C::OFF_B + c0 + i);
                            if (C::RELU) r = fmaxf(r, 0.f);
                            yp[i * plane] = r;
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&ofree[ab]);
        };

        int q = 0;
        for (int ti = 0; ti < ntile; ++ti) {
#pragma unroll 1
            for (int c = 0; c < NCH; ++c, ++q) {
                const int b = q & 1, st = q % NST;
                const float* Wc = Ws + (q % C::NWB) * C::CB;
                mbar_wait(&xfull[st], (q / NST) & 1);
                mbar_wait(&wbar[q % C::NWB], (q / C::NWB) & 1);
                if (q >= 2) mbar_wait(&dfree[b], ((q >> 1) - 1) & 1);            // the MMA that read this operand buffer is complete
                float* Dh = Dbuf + b * 2 * C::DA1;
                dwk_tma_stage<C>(tid, Xb + st * C::BOX, Wc + C::OFF_WD, Wc + C::OFF_BD, Dh, Dh + C::DA1);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) { mbar_arrive(&xfree[st]); mbar_arrive(&dfull[b]); }
                if (c == 0 && ti > 0) epilogue(ti - 1);
            }
        }
        if (ntile > 0) epilogue(ntile - 1);
    }
    __syncthreads();
    if (warp == NWW) {
        __syncwarp();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)C::TCOLS) : "memory");
    }
}

}  // namespace yf
