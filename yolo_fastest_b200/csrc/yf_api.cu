// yf_api.cu — C ABI (include/yf.h) of the B200-native YOLO-Fastest hot path: weight packing,
// the launch plan of fused groups, and the entry points. Kernels live in yf_kernels.cuh / yf_post.cuh.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "../../include/yf.h"
#include "yf_kernels.cuh"
#include "yf_post.cuh"
#include "yf_tc.cuh"
#include "yf_tct.cuh"
#include "yf_wirb.cuh"
#include "yf_tcpw.cuh"
#include "yf_tcpw_tma.cuh"
#include "yf_tcup.cuh"
#include "yf_tcirb2.cuh"
#include "yf_tcdense.cuh"
#include "yf_tcdense2.cuh"
#include "yf_prep.cuh"
#include "yf_jpeg.cuh"
#include "yf_jpeg_enc.cuh"

using namespace yf;

// ---------------------------------------------------------------------------------------------
// canonical parameter order (= forward order of the reference model, yolo_fastest.py:78-148)
// ---------------------------------------------------------------------------------------------
namespace {

struct Spec {
    std::string name;
    int cin, cout, k, groups;
    bool deconv;
    int64_t w_off, b_off;   // offsets (floats) into the host blob
    int64_t w_count() const { return deconv ? (int64_t)cin * cout * k * k : (int64_t)cout * (cin / groups) * k * k; }
};

struct SpecTable {
    std::vector<Spec> specs;
    std::map<std::string, int> index;
    int64_t total = 0;
    void add(const std::string& name, int cin, int cout, int k, int groups = 1, bool deconv = false) {
        Spec s{name, cin, cout, k, groups, deconv, 0, 0};
        s.w_off = total;
        total += s.w_count();
        s.b_off = total;
        total += cout;
        index[name] = (int)specs.size();
        specs.push_back(s);
    }
    void irb(const std::string& name, int io, int mid) {   // BasicResBlock (yolo_fastest.py:52-58)
        add(name + ".conv1", io, mid, 1);
        add(name + ".conv2", mid, mid, 3, mid);
        add(name + ".conv3", mid, io, 1);
    }
    const Spec& get(const std::string& name) const { return specs[index.at(name)]; }
};

// head channels: YoloFastest has num_anchors * (5 + num_cls) (yolo_fastest.py:74-75); YoloFastest_lite multiplies its anchor count
// by the class count first (yolo_fastest.py:240-241)
int head_channels(int num_cls, int num_anchors, int variant) {
    return (variant == YF_VARIANT_LITE ? num_anchors * num_cls : num_anchors) * (5 + num_cls);
}

SpecTable build_specs(int in_ch, int num_cls, int num_anchors, int variant = 0) {
    SpecTable t;
    const int nout = head_channels(num_cls, num_anchors, variant);
    t.add("conv0", in_ch, 8, 3);
    t.add("conv1_2", 8, 8, 1); t.add("conv1_3", 8, 8, 3, 8); t.add("conv1_4", 8, 4, 1);
    t.irb("res1_1", 4, 8);
    t.add("conv1_8", 4, 24, 1); t.add("conv1_9", 24, 24, 3); t.add("conv2_1", 24, 8, 1);
    t.irb("res2_1", 8, 32); t.irb("res2_2", 8, 32);
    t.add("conv2_2", 8, 32, 1); t.add("conv2_3", 32, 32, 3, 32); t.add("conv3_1", 32, 8, 1);
    t.irb("res3_1", 8, 48); t.irb("res3_2", 8, 48);
    t.add("conv3_2", 8, 48, 1); t.add("conv3_3", 48, 48, 3, 48); t.add("conv3_4", 48, 16, 1);
    t.irb("res3_3", 16, 96); t.irb("res3_4", 16, 96); t.irb("res3_5", 16, 96); t.irb("res3_6", 16, 96);
    t.add("conv3_5", 16, 96, 1); t.add("conv3_6", 96, 96, 3, 96); t.add("conv4_1", 96, 24, 1);
    t.irb("res4_1", 24, 136); t.irb("res4_2", 24, 136); t.irb("res4_3", 24, 136); t.irb("res4_4", 24, 136);
    t.add("conv4_2", 24, 136, 1); t.add("conv4_3", 136, 136, 3, 136); t.add("conv5_1", 136, 48, 1);
    t.irb("res5_1", 48, 224); t.irb("res5_2", 48, 224); t.irb("res5_3", 48, 224); t.irb("res5_4", 48, 224);
    t.irb("res5_5", 48, 224);
    t.add("conv5_2", 48, 96, 1);
    t.add("conv5_3", 96, 96, 5, 96); t.add("conv5_4", 96, 128, 1);
    t.add("conv5_5", 128, 128, 5, 128); t.add("conv5_6", 128, 128, 1);
    t.add("head_5", 128, nout, 1);
    t.add("deconv5_1", 96, 96, 2, 1, true);
    t.add("conv4_1_1", 232, 96, 1);
    t.add("conv4_1_2", 96, 96, 5, 96); t.add("conv4_1_3", 96, 96, 1);
    t.add("conv4_1_4", 96, 96, 5, 96); t.add("conv4_1_5", 96, 96, 1);
    t.add("head_4", 96, nout, 1);
    return t;
}

thread_local std::string g_err;

void set_err(std::string* dst, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    (dst ? *dst : g_err) = buf;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------
// tensor map of a group's input (warp-streaming kernels): re-encoded only when the input pointer or the batch changes
struct TmaCache {
    CUtensorMap map;
    const void* ptr = nullptr;
    int B = 0;
    bool u8 = false;
    int box = 0;                 // box shape the map was encoded for (groups whose tile shape depends on the batch; < 0: encode failed)
    bool failed = false;
};

struct GroupArgs {
    TmaCache* tc = nullptr;      // the owning group's tensor-map cache
    int nsm = 148;               // SM count
    int resident = 148;          // persistent grid = CTAs that are co-resident on the device for this group's kernel
    const float* x = nullptr;    // input activation
    const float* x2 = nullptr;   // second input (upcat: low-res tensor)
    float* y = nullptr;          // output activation (or head)
    float* skip = nullptr;       // dual output
    const float* w = nullptr;    // packed weights (device)
    const float* w2 = nullptr;   // second weight block of the same group (the channel-lane kernel's, where a group keeps two engines)
    const DenseSmall* small = nullptr;   // the dense group's small weights (host copy in the ctx: passed to the kernel by value)
    bool pdl = false;            // launch with programmatic stream serialization (set per launch by forward_impl; kernels with pdl_wait() only)
    int Hin = 0, Win = 0, Hout = 0, Wout = 0;
    int headn = 0;
};

// Launch with (pdl) or without the programmatic-stream-serialization attribute (yf_kernels.cuh: pdl_wait). Only kernels that execute
// pdl_wait() before their first activation access may be launched with it.
template <class... KA, class... A>
inline void launch_k(bool pdl, void (*kernel)(KA...), int grid, int block, size_t smem, cudaStream_t st, A&&... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1u : 0u;
    cudaLaunchKernelEx(&cfg, kernel, std::forward<A>(args)...);
}

struct Group {
    int (*occupancy)() = nullptr;                       // resident CTAs per SM of the group's kernel (persistent groups)
    const char* name;                                   // reference attribute producing the group's output
    void (*launch)(const GroupArgs&, const void* xin, bool u8in, int B, cudaStream_t);
    GroupArgs a;
    int out_ch;                                         // channels of y (0 for heads: written to caller memory)
    int64_t w_off;                                      // offset into dev blob (floats)
    TmaCache tcache;
};

struct yf_ctx {
    int variant = 0;                                    // YF_VARIANT_FULL / YF_VARIANT_LITE
    int device = 0, in_ch = 1, num_cls = 3, num_anchors = 3, max_batch = 1, H = 0, W = 0;
    int nout = 0;
    bool weights_loaded = false;
    std::string err;
    SpecTable specs;
    std::vector<Group> groups;
    std::vector<float> host_packed;
    float* d_w = nullptr;
    std::vector<float*> d_act;                          // one buffer per group output
    std::map<std::string, std::pair<float*, int64_t>> taps;   // name -> (buffer, floats per image)
    float* d_skip = nullptr;                            // conv4_2
    float* d_hl = nullptr;                              // internal heads for yf_detect
    float* d_hs = nullptr;
    float* d_x = nullptr;                               // staging for *_host entry points
    unsigned char* d_u8 = nullptr;
    yf_det* d_out = nullptr;
    int out_cap = 0;                                    // max_det capacity of d_out
    int32_t* d_counts = nullptr;
    int32_t* d_status = nullptr;
    // post-process workspace
    int NC = 0;
    yf_det* p_rec = nullptr;
    double* p_conf = nullptr;
    int32_t* p_cls = nullptr;
    int4* p_sbox = nullptr;
    int32_t* p_order = nullptr;
    unsigned char* p_alive = nullptr;
    // double-buffered asynchronous host path (yf_detect_submit_u8 / yf_detect_wait)
    cudaStream_t s_copy = nullptr, s_comp = nullptr, s_back = nullptr;      // H2D of inputs / kernels / D2H of results
    cudaStream_t s_cap = nullptr;                       // graphs are captured here (the caller's stream may be the legacy stream, which cannot capture)
    cudaStream_t s_side = nullptr;                      // small batches: the head_5 branch runs here, beside the upsample branch
    DenseSmall dense_small;                             // conv1_8 / conv2_1 weights and the biases of the dense group (kernel parameter of dense_ta_kernel)
    bool last_forward_forked = false;                   // the last forward ended with an event join: the head kernel is launched the ordinary way
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    unsigned char* sl_u8[2] = {nullptr, nullptr};
    yf_det* sl_out[2] = {nullptr, nullptr};
    int sl_out_cap[2] = {0, 0};
    int32_t* sl_counts[2] = {nullptr, nullptr};
    int32_t* sl_status[2] = {nullptr, nullptr};
    cudaEvent_t sl_in[2] = {nullptr, nullptr}, sl_free[2] = {nullptr, nullptr}, sl_done[2] = {nullptr, nullptr};
    bool sl_used[2] = {false, false};
    // CUDA graphs of forward + head kernel on the library's own fixed buffers (small batches: launch latency dominates)
    std::map<std::string, std::pair<cudaGraphExec_t, int>> graphs;    // key -> (executable graph, kernel launches inside)
    // GPU pre-processing (yf_preprocess_bgr / yf_detect_host_bgr): coefficient tables of the last source size; BGR staging (also of
    // yf_detect_host_frames, whose kernel computes its taps itself)
    PrepTap* prep_tab = nullptr;                        // [W column taps | H row taps]
    int prep_Ho = 0, prep_Wo = 0;
    unsigned char* d_bgr = nullptr;
    size_t bgr_cap = 0;
    int16_t* d_coef = nullptr;                          // JPEG coefficient workspace (128 bytes a block, grow-only, one chunk of files)
    size_t coef_cap = 0;
    unsigned char* d_jframes = nullptr;                 // decoded frames of yf_detect_host_jpeg (grow-only)
    size_t jframes_cap = 0;
    int32_t* d_jstatus = nullptr;                       // per-file decoder status of yf_detect_host_jpeg [max_batch]
    // JPEG encoding (yf_jpeg_enc.cuh), all grow-only: coefficients, bit offsets and bit buffers of one chunk of frames; the header
    // bytes of a call; the files and lengths of yf_encode_host_jpeg before and after packing
    unsigned char* d_jenc = nullptr;
    size_t jenc_cap = 0;
    unsigned char* d_jhdr = nullptr;
    size_t jhdr_cap = 0;
    unsigned char* d_jout = nullptr;
    size_t jout_cap = 0;
    unsigned char* d_jpack = nullptr;
    size_t jpack_cap = 0;
    int64_t* d_jlen = nullptr;
    size_t jlen_cap = 0;
    unsigned char* n_alive = nullptr;                   // yf_nms_sorted_* scratch
    int n_alive_cap = 0;
    int64_t launches = 0;
};

#define CTX_CHECK(ctx)                                         \
    if (!(ctx)) { set_err(nullptr, "null ctx"); return YF_ERR_ARG; }
#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            set_err(&ctx->err, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return YF_ERR_CUDA;                                                               \
        }                                                                                     \
    } while (0)

// ---------------------------------------------------------------------------------------------
// group configurations (tile shapes tuned for the 640x512 / 320x256 maps; any H, W multiple of 32 works)
//        IrbCfg<CIN, CMID, COUT, KS, S, TH, TW, MC, PN1, PN3, RH, NT, MINB, EXPAND, RES, RELU_OUT, DUAL, HEAD>
// ---------------------------------------------------------------------------------------------
// every configuration can be overridden with -DYF_CFG...="..." (tools/tune.py builds variants that way)
#ifndef YF_CFGSTEM
#define YF_CFGSTEM StemCfg<8, 80, 256, 2>
#endif
using CfgStem = YF_CFGSTEM;
using CfgStem3 = StemCfg<8, 40, 256, 2, 3>;          // 3-channel (colour) input: smaller tile, the raw rectangle is three planes
#ifndef YF_CFGRES1
#define YF_CFGRES1 IrbCfg<4, 8, 4, 3, 1, 8, 80, 8, 8, 4, 8, 256, 3, true, true, false, false>
#endif
using CfgRes1 = YF_CFGRES1;
// warp-streaming engine (yf_wirb.cuh) for the thin groups: WirbCfg<CIN, CMID, COUT, S, SPX, NSL, RC, warps, RES, W2 in registers>
#ifndef YF_USE_WIRB
#define YF_USE_WIRB 1    // 0: the thin groups stay on the block-cooperative FFMA engine (comparison arm)
#endif
#ifndef YF_CFGRES1_W
#define YF_CFGRES1_W WirbCfg<4, 8, 4, 1, 4, 8, 6, 12, true, true>
#endif
using CfgRes1W = YF_CFGRES1_W;
#ifndef YF_CFGRES2_W
#define YF_CFGRES2_W WirbCfg<8, 32, 8, 1, 8, 2, 6, 12, true, false>
#endif
using CfgRes2W = YF_CFGRES2_W;
#ifndef YF_CFGDOWN2_W
#define YF_CFGDOWN2_W WirbCfg<8, 32, 8, 2, 4, 2, 8, 12, false, false>
#endif
using CfgDown2W = YF_CFGDOWN2_W;
#ifndef YF_CFGSTEM_W
#define YF_CFGSTEM_W WstemCfg<12>
#endif
using CfgStemW = YF_CFGSTEM_W;

#ifndef YF_CFGDENSE
#define YF_CFGDENSE DenseCfg<8, 40, 4, 128, 3, 2>
#endif
using CfgDense = YF_CFGDENSE;
#ifndef YF_CFGRES2
#define YF_CFGRES2 IrbCfg<8, 32, 8, 3, 1, 8, 40, 16, 8, 4, 8, 128, 4, true, true, false, false>
#endif
using CfgRes2 = YF_CFGRES2;
#ifndef YF_CFGDOWN2
#define YF_CFGDOWN2 IrbCfg<8, 32, 8, 3, 2, 4, 40, 8, 8, 4, 4, 128, 3, true, false, false, false>
#endif
using CfgDown2 = YF_CFGDOWN2;
#ifndef YF_CFGRES3A
#define YF_CFGRES3A IrbCfg<8, 48, 8, 3, 1, 8, 40, 16, 8, 4, 8, 128, 4, true, true, false, false>
#endif
using CfgRes3a = YF_CFGRES3A;
#ifndef YF_CFGWIDE3
#define YF_CFGWIDE3 IrbCfg<8, 48, 16, 3, 1, 8, 40, 24, 8, 8, 8, 256, 2, true, false, false, false>
#endif
using CfgWide3 = YF_CFGWIDE3;
#ifndef YF_CFGRES3B
#define YF_CFGRES3B IrbCfg<16, 96, 16, 3, 1, 8, 40, 16, 8, 8, 8, 256, 2, true, true, false, false>
#endif
using CfgRes3b = YF_CFGRES3B;
// tensor-core (tcgen05, 3xTF32) variant for the wide residual blocks: IrbTcCfg<CIN, CMID, COUT, TH, TW, MC, RH, worker warps, RES>
#ifndef YF_TC3_TH          // tile / chunk / rows-per-item / worker warps of the res3_3..6 instantiation (tools/tc_sweep.sh overrides them)
#define YF_TC3_TH 8
#define YF_TC3_TW 40
#define YF_TC3_MC 32
#define YF_TC3_RH 8
#define YF_TC3_NWW 10
#endif
#ifndef YF_TC3_OCC
#define YF_TC3_OCC 1
#endif
#ifndef YF_TC3_E1ALL
#define YF_TC3_E1ALL false
#endif
#ifndef YF_CFGRES3B_TC
#define YF_CFGRES3B_TC IrbTcCfg<16, 96, 16, YF_TC3_TH, YF_TC3_TW, YF_TC3_MC, YF_TC3_RH, YF_TC3_NWW, true, YF_TC3_E1ALL, YF_TC3_OCC>
#endif
using CfgRes3bTc = YF_CFGRES3B_TC;
#ifndef YF_USE_TCT
#define YF_USE_TCT 1    // 1: res3_3..6 and res4_1..4 run on the channel-lane kernel (yf_tct.cuh) at every batch size (one kernel: results do not depend on the batch)
#endif
#ifndef YF_USE_TCT_A
#define YF_USE_TCT_A 1  // 1: so do the 48-mid-channel groups res3_1, res3_2 and conv3_2 -> conv3_4
#endif
// IrbTtCfg<CIN, CMID, COUT, tile height (x 8 columns), RES, TMEM lane quarter of channel 128, CTAs per SM, depthwise stride, dual output, ReLU after the projection>
using CfgRes3bTt = IrbTtCfg<16, 96, 16, 16, true>;
using CfgRes4Tt = IrbTtCfg<24, 136, 24, 8, true, 2>;
#ifndef YF_TCT_A_TH
#define YF_TCT_A_TH 16      // measured: 8-row tiles at two CTAs per SM are no faster (0.137 ms either way)
#define YF_TCT_A_OCC 1
#endif
using CfgRes3aTt = IrbTtCfg<8, 48, 8, YF_TCT_A_TH, true, 0, YF_TCT_A_OCC>;
using CfgWide3Tt = IrbTtCfg<8, 48, 16, YF_TCT_A_TH, false, 0, YF_TCT_A_OCC>;
using CfgDown3Tt = IrbTtCfg<16, 96, 24, 8, false, 0, 1, 2>;          // conv3_5 -> conv3_6 (stride 2) -> conv4_1
using CfgDown4Tt = IrbTtCfg<24, 136, 48, 4, false, 1, 1, 2, true, true>;    // conv4_2 (also the neck's skip tensor) -> conv4_3 (stride 2) -> conv5_1
#ifndef YF_CFGRES4_TC
#define YF_CFGRES4_TC IrbTcCfg<24, 136, 24, 8, 20, 32, 4, 10, true, true>
#endif
using CfgRes4Tc = YF_CFGRES4_TC;
// res4 maps are 1/16 of the input: their rows are a multiple of 16 bytes (what a TMA tensor map needs) only when the input width is a
// multiple of 64. Other widths (416 -> 26 columns) keep the pixel-lane kernel; the group holds both weight blocks (GroupArgs::w, w2).
#ifndef YF_USE_TC
#define YF_USE_TC 1     // 1: res3_3..6 and res4_1..4 run on the tcgen05 kernel (yf_tc.cuh); 0: everything on the FFMA engine (libyf_b200_ffma.so)
#endif
#ifndef YF_CFGDOWN3
#define YF_CFGDOWN3 IrbCfg<16, 96, 24, 3, 2, 4, 40, 16, 8, 8, 4, 256, 2, true, false, false, false>
#endif
using CfgDown3 = YF_CFGDOWN3;
#ifndef YF_CFGRES4
#define YF_CFGRES4 IrbCfg<24, 136, 24, 3, 1, 8, 40, 16, 8, 8, 8, 256, 2, true, true, false, false>
#endif
using CfgRes4 = YF_CFGRES4;
#ifndef YF_CFGDOWN4
#define YF_CFGDOWN4 IrbCfg<24, 136, 48, 3, 2, 2, 20, 16, 8, 8, 2, 128, 4, true, false, true, true>
#endif
using CfgDown4 = YF_CFGDOWN4;
#ifndef YF_CFGRES5
#define YF_CFGRES5 IrbCfg<48, 224, 48, 3, 1, 8, 20, 16, 8, 8, 8, 256, 2, true, true, false, false>
#endif
using CfgRes5 = YF_CFGRES5;
#ifndef YF_CFGPW52
#define YF_CFGPW52 PwCfg<48, 96, 80, 8, 256, true>
#endif
using CfgPw52 = YF_CFGPW52;
using CfgLite34 = PwPwCfg<8, 48, 16, 128>;          // YoloFastest_lite: conv3_2 -> conv3_4 without the depthwise conv3_3
#ifndef YF_CFGNECKS1
#define YF_CFGNECKS1 IrbCfg<96, 96, 128, 5, 1, 8, 20, 48, 4, 8, 4, 640, 1, false, false, false, false>
#endif
using CfgNeckS1 = YF_CFGNECKS1;
#ifndef YF_CFGNECKS2
#define YF_CFGNECKS2 IrbCfg<128, 128, 128, 5, 1, 8, 20, 32, 4, 8, 4, 640, 1, false, false, false, false, 1>
#endif
using CfgNeckS2 = YF_CFGNECKS2;
#ifndef YF_CFGUPCAT
#define YF_CFGUPCAT UpCatCfg<8, 20, 16, 4, 256, 2>
#endif
using CfgUpCat = YF_CFGUPCAT;
#ifndef YF_CFGNECKL1
#define YF_CFGNECKL1 IrbCfg<96, 96, 96, 5, 1, 4, 40, 32, 4, 8, 4, 256, 2, false, false, false, false>
#endif
using CfgNeckL1 = YF_CFGNECKL1;
#ifndef YF_CFGNECKL2
#define YF_CFGNECKL2 IrbCfg<96, 96, 96, 5, 1, 4, 40, 16, 4, 8, 4, 256, 2, false, false, false, false, 1>
#endif
using CfgNeckL2 = YF_CFGNECKL2;
// tensor-core depthwise -> wide 1x1 pairs of the neck: DwPwTcCfg<C, N, KS, TH, TW, MC, RH, worker warps, RELU>
#ifndef YF_CFGNECKS1_TC
#define YF_CFGNECKS1_TC DwPwTcCfg<96, 128, 5, 16, 20, 16, 4, 10, false>
#endif
using CfgNeckS1Tc = YF_CFGNECKS1_TC;
#ifndef YF_CFGNECKL1_TC
#define YF_CFGNECKL1_TC DwPwTcCfg<96, 96, 5, 8, 40, 16, 4, 10, false>
#endif
using CfgNeckL1Tc = YF_CFGNECKL1_TC;
// head groups with at most 32 output channels (the shipped 3-class models: 24): depthwise 5x5 -> composed 1x1, N = 32
#ifndef YF_CFGNECKS2_TC
#define YF_CFGNECKS2_TC DwPwTcCfg<128, 32, 5, 16, 20, 16, 4, 10, false, true>
#endif
using CfgNeckS2Tc = YF_CFGNECKS2_TC;
#ifndef YF_CFGNECKL2_TC
#define YF_CFGNECKL2_TC DwPwTcCfg<96, 32, 5, 8, 40, 16, 4, 10, false, true>
#endif
using CfgNeckL2Tc = YF_CFGNECKL2_TC;
static bool heads_on_tc(int nout) { return YF_USE_TC && nout <= 32; }
using CfgUpCatTc = UpCatTcCfg<10>;
using CfgDenseTc = DenseTcCfg<12>;
#ifndef YF_DENSE_TC
#define YF_DENSE_TC YF_USE_TC       // the dense 3x3 group on tcgen05
#endif
#ifndef YF_RES5_TC
#define YF_RES5_TC YF_USE_TC        // res5_* on tcgen05
#endif
// widest residual blocks on the chunked tensor-core engine: IrbTc2Cfg<CIN, CMID, COUT, TH, TW, N halves, RH, worker warps, RES>
#ifndef YF_CFGRES5_TC
#define YF_CFGRES5_TC IrbTc2Cfg<48, 224, 48, 8, 20, 2, 2, 10, true>
#endif
using CfgRes5Tc = YF_CFGRES5_TC;
// Small-batch (latency) variants: the same kernels and the same packed weights on half-height tiles. At batch 1 the low-resolution
// maps give a handful of tiles (res5: 2, res4: 8, res3: 16 of the throughput shape), i.e. most SMs idle while one tile's step chain
// runs; halving the tile halves that chain. Chosen per launch when the throughput tiling would leave more than half of the SMs idle.
using CfgRes5TcS = IrbTc2Cfg<48, 224, 48, 4, 20, 2, 2, 10, true>;
using CfgRes4TcS = IrbTcCfg<24, 136, 24, 4, 20, 32, 4, 10, true, true>;
using CfgRes3bTcS = IrbTcCfg<16, 96, 16, 4, 40, 32, 4, 10, true, YF_TC3_E1ALL>;
using CfgRes5TcXS = IrbTc2Cfg<48, 224, 48, 2, 20, 2, 2, 10, true>;          // quarter height: when even the half-height tiles leave 3/4 of the SMs idle
// Narrow-map variants: tile widths that fit the 1/16 and 1/32 maps of the 320x256 input (20 and 10 columns) - the throughput shapes
// (40 / 20 columns wide) would compute half or three quarters of every tile outside the image. Same packed weights again.
using CfgRes5TcN = IrbTc2Cfg<48, 224, 48, 8, 12, 2, 2, 10, true>;
using CfgNeckS1TcN = DwPwTcCfg<96, 128, 5, 8, 12, 16, 4, 10, false>;
using CfgNeckS2TcN = DwPwTcCfg<128, 32, 5, 8, 12, 16, 4, 10, false, true>;
using CfgNeckL1TcN = DwPwTcCfg<96, 96, 5, 8, 20, 16, 4, 10, false>;
using CfgNeckL2TcN = DwPwTcCfg<96, 32, 5, 8, 20, 16, 4, 10, false, true>;
using CfgDown3N = IrbCfg<16, 96, 24, 3, 2, 4, 20, 16, 8, 8, 4, 256, 2, true, false, false, false>;
using CfgDown4N = IrbCfg<24, 136, 48, 3, 2, 2, 12, 16, 8, 8, 2, 128, 4, true, false, true, true>;
using CfgNeckL1TcS = DwPwTcCfg<96, 96, 5, 4, 20, 16, 4, 10, false>;
using CfgNeckL2TcS = DwPwTcCfg<96, 32, 5, 4, 20, 16, 4, 10, false, true>;
using CfgNeckS1TcS = DwPwTcCfg<96, 128, 5, 4, 20, 16, 4, 10, false>;
using CfgNeckS2TcS = DwPwTcCfg<128, 32, 5, 4, 20, 16, 4, 10, false, true>;
using CfgRes3bTcXS = IrbTcCfg<16, 96, 16, 2, 40, 32, 2, 10, true, YF_TC3_E1ALL>;
using CfgRes4TcXS = IrbTcCfg<24, 136, 24, 2, 20, 32, 2, 10, true, true>;
// the tensor-core upsample+concat kernel moves the skip tensor with 128-bit loads: it needs the 1/16-resolution map to be a
// multiple of 4 wide and even in height (true for the shipped 512x640 / 256x320 models; 416x416 falls back to upcat_kernel)
static bool upcat_on_tc(int H, int W) { return YF_USE_TC && ((W / 16) % 4 == 0) && ((H / 16) % 2 == 0); }

namespace {

template <class C>
void launch_irb(const GroupArgs& g, const void*, bool, int B, cudaStream_t st) {
    using G = typename C::G;
    const int tx = cdiv(g.Wout, G::TW), ty = cdiv(g.Hout, G::TH);
    const int total = B * tx * ty;
    const int grid = total < g.resident ? total : g.resident;     // persistent: every CTA resident, loops over tiles
    irb_kernel<C><<<grid, C::NT, C::SMEM_BYTES, st>>>(g.x, g.y, g.skip, g.w, g.Hin, g.Win, g.Hout, g.Wout, tx, ty, total, g.headn);
}
template <class CB, class CN>
void launch_irb_auto(const GroupArgs& g, const void* x, bool u8, int B, cudaStream_t st) {      // CN: the narrow-map tile shape
    static_assert(CB::CB == CN::CB && CB::OFF_B2 == CN::OFF_B2 && CB::MC == CN::MC, "both tile shapes read the same packed weights");
    const int big = B * cdiv(g.Wout, CB::G::TW) * cdiv(g.Hout, CB::G::TH);
    if (g.Wout <= CN::G::TW || 2 * big <= g.nsm) launch_irb<CN>(g, x, u8, B, st);      // narrow map, or a small batch: more, smaller tiles
    else launch_irb<CB>(g, x, u8, B, st);
}
template <class K>
int occ_of(K kernel, int nt, int smem) {
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, nt, smem) != cudaSuccess || n < 1) n = 1;
    return n;
}
template <class C> int occ_irb() { return occ_of(irb_kernel<C>, C::NT, C::SMEM_BYTES); }
int occ_stem() { return occ_of(stem_kernel<CfgStem, false>, CfgStem::NT, CfgStem::SMEM_BYTES); }
int occ_stem3() { return occ_of(stem_kernel<CfgStem3, false>, CfgStem3::NT, CfgStem3::SMEM_BYTES); }
int occ_dense() { return occ_of(dense_kernel<CfgDense>, CfgDense::NT, CfgDense::SMEM_BYTES); }
int occ_upcat() { return occ_of(upcat_kernel<CfgUpCat>, CfgUpCat::NT, CfgUpCat::SMEM_BYTES); }
int occ_upcat_tc() { return occ_of(upcat_tc_kernel<CfgUpCatTc>, CfgUpCatTc::NT, CfgUpCatTc::SMEM_BYTES); }
void launch_upcat_tc(const GroupArgs& g, const void*, bool, int B, cudaStream_t st) {
    using C = CfgUpCatTc;
    const int tx = cdiv(g.Wout, C::TW), ty = cdiv(g.Hout, C::TH);
    const int total = B * tx * ty;
    const int grid = total < g.resident ? total : g.resident;
    launch_k(g.pdl, upcat_tc_kernel<C>, grid, C::NT, C::SMEM_BYTES, st, g.x, g.x2, g.y, g.w, g.Hout, g.Wout, tx, ty, total);
}

// warp-streaming groups: one warp per (image, band of R output rows, strip of OW columns). The band height is chosen per launch:
// it trades the 2 halo rows per band against the load balance of units over the resident warps.
template <class C>
int wirb_band_rows(int B, int Hout, int Wout, int warps) {
    const int nstrips = cdiv(Wout, C::OW);
    long long best_cost = -1;
    int best_R = 1;
    for (int nch = 1; nch <= 16; ++nch) {
        const int R = C::S == 1 ? nch * C::RC - 2 : (nch * C::RC - 1) / 2;      // the tallest band whose input rows fill nch boxes
        if (R < 1) continue;
        const long long units = (long long)B * nstrips * cdiv(Hout, R);
        const long long cost = ((units + warps - 1) / warps) * (nch * C::RC + 2);  // box rows per warp (+ per-unit set-up)
        if (best_cost < 0 || cost <= best_cost) { best_cost = cost; best_R = R; }
        if (R >= Hout) break;
    }
    return best_R;
}
template <class C>
void launch_wirb(const GroupArgs& g, const void*, bool, int B, cudaStream_t st) {
    TmaCache* tc = g.tc;
    if (tc->ptr != g.x || tc->B != B) {
        tc->failed = tma_make_map4(&tc->map, g.x, 4, B, C::CIN, g.Hin, g.Win, C::XW, C::RC, C::CIN) != 0;
        tc->ptr = g.x; tc->B = B;
    }
    if (g.Wout % C::SPX) tc->failed = true;               // the edge masks assume whole strips (true for every H, W multiple of 32)
    if (tc->failed) return;
    const int R = wirb_band_rows<C>(B, g.Hout, g.Wout, g.nsm * C::NW);
    const int nstrips = cdiv(g.Wout, C::OW), nbands = cdiv(g.Hout, R);
    const int total = B * nstrips * nbands;
    const int grid = std::min(g.nsm, cdiv(total, C::NW));
    launch_k(g.pdl, wirb_kernel<C>, grid, C::NW * 32, C::SMEM_BYTES, st, tc->map, g.y, g.w, g.Hin, g.Win, g.Hout, g.Wout, R, nstrips, nbands, total);
}
// stem group on the warp-streaming engine (single-channel input): the raw image is the TMA tensor, fp32 or uint8
template <class C>
void launch_wstem(const GroupArgs& g, const void* xin, bool u8in, int B, cudaStream_t st) {
    TmaCache* tc = g.tc;
    if (tc->ptr != xin || tc->B != B || tc->u8 != u8in) {
        tc->failed = (u8in ? tma_make_map4(&tc->map, xin, 1, B, 1, g.Hin, g.Win, C::RAWWU, C::RAWH, 1)
                           : tma_make_map4(&tc->map, xin, 4, B, 1, g.Hin, g.Win, C::RAWW, C::RAWH, 1)) != 0;
        tc->ptr = xin; tc->B = B; tc->u8 = u8in;
    }
    if (g.Wout % C::SPX) tc->failed = true;
    if (tc->failed) return;
    const int R = wirb_band_rows<C>(B, g.Hout, g.Wout, g.nsm * C::NW);
    const int nstrips = cdiv(g.Wout, C::OW), nbands = cdiv(g.Hout, R);
    const int total = B * nstrips * nbands;
    const int grid = std::min(g.nsm, cdiv(total, C::NW));
    if (u8in) launch_k(g.pdl, wstem_kernel<C, true>, grid, C::NW * 32, C::template smem_bytes<true>(), st, tc->map, g.y, g.w, g.Hin, g.Win, g.Hout, g.Wout, R, nstrips, nbands, total);
    else launch_k(g.pdl, wstem_kernel<C, false>, grid, C::NW * 32, C::template smem_bytes<false>(), st, tc->map, g.y, g.w, g.Hin, g.Win, g.Hout, g.Wout, R, nstrips, nbands, total);
}
template <class C>
cudaError_t init_wstem() {
    cudaError_t e = cudaFuncSetAttribute(wstem_kernel<C, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::template smem_bytes<true>());
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(wstem_kernel<C, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::template smem_bytes<false>());
}

template <class C>
cudaError_t init_wirb() { return cudaFuncSetAttribute(wirb_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES); }

// The depthwise 5x5 -> 1x1 groups take their input by tensor-tile TMA (dwpw_tma_kernel) where the map's rows are a multiple of 16 bytes
// and the tensor map encodes; otherwise, and in a -DYF_DWPW_TMA=0 build, the cp.async kernel dwpw_tc_kernel. Both read the same packed
// weights and give the same bits.
#ifndef YF_DWPW_TMA
#define YF_DWPW_TMA 1
#endif
template <class C>
void launch_dwpwtc(const GroupArgs& g, const void*, bool, int B, cudaStream_t st) {
    using G = typename C::G;
    using T = DwPwTmaCfg<C>;
    const int tx = cdiv(g.Wout, G::TW), ty = cdiv(g.Hout, G::TH);
    const int total = B * tx * ty;
    const int grid = total < g.resident ? total : g.resident;
    const int nout = g.headn > 0 ? g.headn : C::N;
    bool tma = YF_DWPW_TMA && g.Wout % 4 == 0;
    if (tma) {
        TmaCache* tc = g.tc;
        const int box = T::BW * 1024 + T::BH;
        if (tc->ptr != g.x || tc->B != B || (tc->box != box && tc->box != -box)) {
            // an encode failure selects the cp.async kernel for this input (recorded as -box), it is not a forward error
            const bool ok = tma_make_map4(&tc->map, g.x, 4, B, C::C, g.Hout, g.Wout, T::BW, T::BH, C::MC) == 0;
            tc->ptr = g.x; tc->B = B; tc->box = ok ? box : -box;
        }
        tma = tc->box == box;
    }
    if (tma) launch_k(g.pdl, dwpw_tma_kernel<T>, grid, T::NT, T::SMEM_BYTES, st, g.tc->map, g.y, g.w, g.Hout, g.Wout, tx, ty, total, nout);
    else launch_k(g.pdl, dwpw_tc_kernel<C>, grid, C::NT, C::SMEM_BYTES, st, g.x, g.y, g.w, g.Hout, g.Wout, tx, ty, total, nout);
}
template <class CB, class CS, class CN>
void launch_dwpwtc_auto(const GroupArgs& g, const void* x, bool u8, int B, cudaStream_t st) {      // CS: small batches, CN: narrow maps
    static_assert(CB::WFLOATS == CS::WFLOATS && CB::CB == CS::CB && CB::WFLOATS == CN::WFLOATS && CB::CB == CN::CB, "all tile shapes read the same packed weights");
    const int big = B * cdiv(g.Wout, CB::G::TW) * cdiv(g.Hout, CB::G::TH);
    if (g.Wout <= CN::G::TW) launch_dwpwtc<CN>(g, x, u8, B, st);
    else if (2 * big <= g.nsm) launch_dwpwtc<CS>(g, x, u8, B, st);
    else launch_dwpwtc<CB>(g, x, u8, B, st);
}
template <class C> int occ_dwpwtc() {
    return std::min(occ_of(dwpw_tc_kernel<C>, C::NT, C::SMEM_BYTES), occ_of(dwpw_tma_kernel<DwPwTmaCfg<C>>, DwPwTmaCfg<C>::NT, DwPwTmaCfg<C>::SMEM_BYTES));
}
template <class C>
cudaError_t init_dwpwtc() {
    const cudaError_t e = cudaFuncSetAttribute(dwpw_tc_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(dwpw_tma_kernel<DwPwTmaCfg<C>>, cudaFuncAttributeMaxDynamicSharedMemorySize, DwPwTmaCfg<C>::SMEM_BYTES);
}

template <class C>
void launch_irbtc2(const GroupArgs& g, const void*, bool, int B, cudaStream_t st) {
    using G = typename C::G;
    const int tx = cdiv(g.Wout, G::TW), ty = cdiv(g.Hout, G::TH);
    const int total = B * tx * ty;
    const int grid = total < g.resident ? total : g.resident;
    launch_k(g.pdl, irbtc2_kernel<C>, grid, C::NT, C::SMEM_BYTES, st, g.x, g.y, g.w, g.Hout, g.Wout, tx, ty, total);
}
// big tiles unless they would occupy less than half of the SMs (small batches): then the half-height variant
template <class CB, class CS>
void launch_irbtc2_auto(const GroupArgs& g, const void* x, bool u8, int B, cudaStream_t st) {
    const int big = B * cdiv(g.Wout, CB::G::TW) * cdiv(g.Hout, CB::G::TH);
    if (g.Wout <= CfgRes5TcN::G::TW) launch_irbtc2<CfgRes5TcN>(g, x, u8, B, st);
    else if (4 * big <= g.nsm) launch_irbtc2<CfgRes5TcXS>(g, x, u8, B, st);
    else if (2 * big <= g.nsm) launch_irbtc2<CS>(g, x, u8, B, st);
    else launch_irbtc2<CB>(g, x, u8, B, st);
}
template <class C> int occ_irbtc2() { return occ_of(irbtc2_kernel<C>, C::NT, C::SMEM_BYTES); }
template <class C>
cudaError_t init_irbtc2() { return cudaFuncSetAttribute(irbtc2_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES); }

template <class C>
void launch_irbtc(const GroupArgs& g, const void*, bool, int B, cudaStream_t st) {
    using G = typename C::G;
    const int tx = cdiv(g.Wout, G::TW), ty = cdiv(g.Hout, G::TH);
    const int total = B * tx * ty;
    const int grid = total < g.resident ? total : g.resident;
    irbtc_kernel<C><<<grid, C::NT, C::SMEM_BYTES, st>>>(g.x, g.y, g.w, g.Hout, g.Wout, tx, ty, total);
}
template <class CB, class CS, class CXS>
void launch_irbtc_auto(const GroupArgs& g, const void* x, bool u8, int B, cudaStream_t st) {
    static_assert(CB::WFLOATS == CS::WFLOATS && CB::CB == CS::CB && CB::OFF_B2 == CS::OFF_B2 && CB::WFLOATS == CXS::WFLOATS && CB::CB == CXS::CB,
                  "all tile shapes read the same packed weights");
    const int big = B * cdiv(g.Wout, CB::G::TW) * cdiv(g.Hout, CB::G::TH);
    if (4 * big <= g.nsm) launch_irbtc<CXS>(g, x, u8, B, st);
    else if (2 * big <= g.nsm) launch_irbtc<CS>(g, x, u8, B, st);
    else launch_irbtc<CB>(g, x, u8, B, st);
}
template <class C>
void launch_irbt(const GroupArgs& g, const void*, bool, int B, cudaStream_t st, int64_t w_off = 0) {
    TmaCache* tc = g.tc;
    if (tc->ptr != g.x || tc->B != B) {
        tc->failed = tma_make_map4(&tc->map, g.x, 4, B, C::CIN, g.Hin, g.Win, C::RW, C::HR, C::CIN) != 0;
        tc->ptr = g.x; tc->B = B;
    }
    if (tc->failed) return;
    const int tx = cdiv(g.Wout, C::TW), ty = cdiv(g.Hout, C::TH);
    const int total = B * tx * ty;
    const int grid = total < g.nsm * C::OCC ? total : g.nsm * C::OCC;
    launch_k(g.pdl, irbt_kernel<C>, grid, C::NT, C::SMEM_BYTES, st, tc->map, g.x, g.y, g.skip, g.w + w_off, g.Hin, g.Win, g.Hout, g.Wout, tx, ty, total);
}
template <class C>
cudaError_t init_irbt() { return cudaFuncSetAttribute(irbt_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES); }
template <class C> void launch_irbt0(const GroupArgs& g, const void* x, bool u8, int B, cudaStream_t st) { launch_irbt<C>(g, x, u8, B, st, 0); }
// res4: the channel-lane kernel where the map's rows can be a TMA tensor (shape only: the choice never depends on the batch)
template <class CT, class CB, class CS, class CXS>
void launch_res4_auto(const GroupArgs& g, const void* x, bool u8, int B, cudaStream_t st) {
    if (g.Wout % 4 == 0) launch_irbt<CT>(g, x, u8, B, st, g.w2 - g.w);
    else launch_irbtc_auto<CB, CS, CXS>(g, x, u8, B, st);
}
// conv5_1's input is a 1/16 map as well: same rule, same two weight blocks
template <class CT, class CB, class CN>
void launch_down4_auto(const GroupArgs& g, const void* x, bool u8, int B, cudaStream_t st) {
    if (g.Win % 4 == 0) launch_irbt<CT>(g, x, u8, B, st, g.w2 - g.w);
    else launch_irb_auto<CB, CN>(g, x, u8, B, st);
}
template <class C> int occ_irbt() { return occ_of(irbt_kernel<C>, C::NT, C::SMEM_BYTES); }
template <class C> int occ_irbtc() { return occ_of(irbtc_kernel<C>, C::NT, C::SMEM_BYTES); }
template <class C>
cudaError_t init_irbtc() { return cudaFuncSetAttribute(irbtc_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES); }

template <class C>
cudaError_t init_irb() { return cudaFuncSetAttribute(irb_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES); }

template <class C>
void launch_stem(const GroupArgs& g, const void* xin, bool u8in, int B, cudaStream_t st) {
    using G = typename C::G;
    const int tx = cdiv(g.Wout, G::TW), ty = cdiv(g.Hout, G::TH);
    const int total = B * tx * ty;
    const int grid = total < g.resident ? total : g.resident;
    if (u8in) stem_kernel<C, true><<<grid, C::NT, C::SMEM_BYTES, st>>>(xin, g.y, g.w, g.Hin, g.Win, g.Hout, g.Wout, tx, ty, total);
    else stem_kernel<C, false><<<grid, C::NT, C::SMEM_BYTES, st>>>(xin, g.y, g.w, g.Hin, g.Win, g.Hout, g.Wout, tx, ty, total);
}
int occ_dense_tc() { return occ_of(dense_tc_kernel<CfgDenseTc>, CfgDenseTc::NT, CfgDenseTc::SMEM_BYTES); }
void launch_dense_tc(const GroupArgs& g, const void*, bool, int B, cudaStream_t st) {
    using C = CfgDenseTc;
    const int tx = cdiv(g.Wout, C::TW), ty = cdiv(g.Hout, C::TH);
    const int total = B * tx * ty;
    const int grid = total < g.resident ? total : g.resident;
    launch_k(g.pdl, dense_tc_kernel<C>, grid, C::NT, C::SMEM_BYTES, st, g.x, g.y, g.w, g.Hin, g.Win, g.Hout, g.Wout, tx, ty, total);
}
// the same group with the A operand in tensor memory (yf_tcdense2.cuh); same packed weights
#ifndef YF_DENSE_TA
#define YF_DENSE_TA 1
#endif
int occ_dense_ta() { return occ_of(dense_ta_kernel<DenseTaCfg>, DenseTaCfg::NT, DenseTaCfg::SMEM_BYTES); }
void launch_dense_ta(const GroupArgs& g, const void*, bool, int B, cudaStream_t st) {
    using C = DenseTaCfg;
    TmaCache* tc = g.tc;
    if (tc->ptr != g.x || tc->B != B) {
        tc->failed = tma_make_map4(&tc->map, g.x, 4, B, 4, g.Hin, g.Win, C::XW, C::RH, 4) != 0;
        tc->ptr = g.x; tc->B = B;
    }
    if (tc->failed) return;
    const int tx = cdiv(g.Wout, C::TW), ty = cdiv(g.Hout, C::TH);
    const int total = B * tx * ty;
    const int grid = total < g.resident ? total : g.resident;
    launch_k(g.pdl, dense_ta_kernel<C>, grid, C::NT, C::SMEM_BYTES, st, tc->map, g.y, g.w, *g.small, g.Hin, g.Win, g.Hout, g.Wout, tx, ty, total);
}
void launch_dense(const GroupArgs& g, const void*, bool, int B, cudaStream_t st) {
    using C = CfgDense;
    using G = C::G;
    const int tx = cdiv(g.Wout, G::TW), ty = cdiv(g.Hout, G::TH);
    const int total = B * tx * ty;
    const int grid = total < g.resident ? total : g.resident;
    dense_kernel<C><<<grid, C::NT, C::SMEM_BYTES, st>>>(g.x, g.y, g.w, g.Hin, g.Win, g.Hout, g.Wout, tx, ty, total);
}
void launch_pw52(const GroupArgs& g, const void*, bool, int B, cudaStream_t st) {
    using C = CfgPw52;
    const int HW = g.Hin * g.Win;
    const int tiles = cdiv(HW, C::PIXT);
    launch_k(g.pdl, pw_kernel<C>, B * tiles, C::NT, C::SMEM_BYTES, st, g.x, g.y, g.w, HW, tiles);
}
void launch_lite34(const GroupArgs& g, const void*, bool, int B, cudaStream_t st) {
    using C = CfgLite34;
    const int HW = g.Hin * g.Win;
    const long long groups = (long long)B * (HW / 4);
    const int grid = (int)std::min<long long>((groups + C::NT - 1) / C::NT, (long long)g.nsm * 8);
    pwpw_kernel<C><<<grid, C::NT, 0, st>>>(g.x, g.y, g.w, HW, groups);
}
void launch_upcat(const GroupArgs& g, const void*, bool, int B, cudaStream_t st) {
    using C = CfgUpCat;
    const int tx = cdiv(g.Wout, C::TW), ty = cdiv(g.Hout, C::TH);
    const int total = B * tx * ty;
    const int grid = total < g.resident ? total : g.resident;
    upcat_kernel<C><<<grid, C::NT, C::SMEM_BYTES, st>>>(g.x, g.x2, g.y, g.w, g.Hout, g.Wout, tx, ty, total);
}

// ---- packing -------------------------------------------------------------------------------
struct Folded {
    const float* blob;
    const SpecTable* t;
    const float* w(const std::string& n) const { return blob + t->get(n).w_off; }
    const float* b(const std::string& n) const { return blob + t->get(n).b_off; }
};

void pad4(std::vector<float>& v) { while (v.size() % 4) v.push_back(0.f); }

// expand name (or "" when !EXPAND), depthwise name, project name, optional head name
template <class C>
int64_t pack_irb(std::vector<float>& out, const Folded& f, const std::string& n1, const std::string& nd,
                 const std::string& n2, const std::string& nh, int headn) {
    pad4(out);
    const int64_t off = (int64_t)out.size();
    const int headp = rup(headn, 4);
    out.resize(off + (C::HEADC ? C::OFF_WH + C::CMIDP * headp + headp : C::OFF_B2 + C::COUT), 0.f);
    float* o = out.data() + off;
    for (int c = 0; c < C::NCHUNK; ++c) {
        float* cb = o + (int64_t)c * C::CB;
        for (int ml = 0; ml < C::MC; ++ml) {
            const int m = c * C::MC + ml;
            if (m >= C::CMID) continue;   // zero padding of the mid channels
            if (C::EXPAND) {
                for (int k = 0; k < C::CIN; ++k) cb[C::OFF_W1 + k * C::MC + ml] = f.w(n1)[m * C::CIN + k];
                cb[C::OFF_B1 + ml] = f.b(n1)[m];
            }
            for (int t = 0; t < C::KK; ++t) cb[C::OFF_WD + ml * C::KK + t] = f.w(nd)[m * C::KK + t];
            cb[C::OFF_BD + ml] = f.b(nd)[m];
            if (!C::HEADC)
                for (int n = 0; n < C::COUT; ++n) cb[C::OFF_W2 + ml * C::COUT + n] = f.w(n2)[n * C::CMID + m];
        }
    }
    if (!C::HEADC) {
        for (int n = 0; n < C::COUT; ++n) o[C::OFF_B2 + n] = f.b(n2)[n];
    } else {
        // n2 (conv5_6 / conv4_1_5: BN-folded 1x1, NO activation, yolo_fastest.py:136,146) followed by the biased head conv nh
        // (:138,148) are two linear maps; compose them in double precision:  Wh' = Wh . W2,  bh' = Wh . b2 + bh
        float* wh = o + C::OFF_WH;
        float* bh = wh + C::CMIDP * headp;
        for (int n = 0; n < headn; ++n) {
            for (int m = 0; m < C::CMID; ++m) {
                double a = 0.0;
                for (int k = 0; k < C::COUT; ++k) a += (double)f.w(nh)[n * C::COUT + k] * (double)f.w(n2)[k * C::CMID + m];
                wh[m * headp + n] = (float)a;
            }
            double b = (double)f.b(nh)[n];
            for (int k = 0; k < C::COUT; ++k) b += (double)f.w(nh)[n * C::COUT + k] * (double)f.b(n2)[k];
            bh[n] = (float)b;
        }
    }
    return off;
}

inline float tf32_rna_host(float v) {      // cvt.rna.tf32.f32: round to nearest (ties away) at 10 mantissa bits
    uint32_t u;
    memcpy(&u, &v, 4);
    u = (u + 0x1000u) & 0xFFFFE000u;
    memcpy(&v, &u, 4);
    return v;
}
// weights of a tensor-core block: K-major core-matrix layout [n/8][k/4][n%8][k%4], split into hi = tf32(w) and lo = w - hi
inline void put_kmajor_split(float* hi, float* lo, int n, int k, int K, float w) {
    const int idx = ((n >> 3) * (K / 4) + (k >> 2)) * 32 + (n & 7) * 4 + (k & 3);
    const float h = tf32_rna_host(w);
    hi[idx] = h;
    lo[idx] = tf32_rna_host(w - h);      // rounded, not left to the tensor core's truncation (which would bias every product the same way)
}

// warp-streaming group: [W1: CIN x CMID][b1][Wd: 9 x CMID][bd][W2: COUT x CMID][b2]
template <class C>
int64_t pack_wirb(std::vector<float>& out, const Folded& f, const std::string& n1, const std::string& nd, const std::string& n2) {
    pad4(out);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    for (int m = 0; m < C::CMID; ++m) {
        for (int k = 0; k < C::CIN; ++k) o[C::OFF_W1 + k * C::CMID + m] = f.w(n1)[m * C::CIN + k];
        o[C::OFF_B1 + m] = f.b(n1)[m];
        for (int t = 0; t < 9; ++t) o[C::OFF_WD + t * C::CMID + m] = f.w(nd)[m * 9 + t];
        o[C::OFF_BD + m] = f.b(nd)[m];
        for (int n = 0; n < C::COUT; ++n) o[C::OFF_W2 + n * C::CMID + m] = f.w(n2)[n * C::CMID + m];
    }
    for (int n = 0; n < C::COUT; ++n) o[C::OFF_B2 + n] = f.b(n2)[n];
    return off;
}

// head group on the tensor-core depthwise -> 1x1 kernel: n2 (linear 1x1) and nh (biased head conv) composed as in pack_irb
template <class C>
int64_t pack_dwpwtc_head(std::vector<float>& out, const Folded& f, const std::string& nd, const std::string& n2, const std::string& nh, int mid, int headn) {
    pad4(out);
    while (out.size() % 32) out.push_back(0.f);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    for (int c = 0; c < C::NCHUNK; ++c) {
        float* cb = o + (int64_t)c * C::CB;
        for (int ml = 0; ml < C::MC; ++ml) {
            const int m = c * C::MC + ml;
            for (int t = 0; t < C::KK; ++t) cb[C::OFF_WD + ml * C::KK + t] = f.w(nd)[m * C::KK + t];
            cb[C::OFF_BD + ml] = f.b(nd)[m];
            for (int n = 0; n < headn; ++n) {
                double a = 0.0;
                for (int k = 0; k < mid; ++k) a += (double)f.w(nh)[n * mid + k] * (double)f.w(n2)[k * C::C + m];
                put_kmajor_split(cb + C::OFF_WH, cb + C::OFF_WL, n, ml, C::MC, (float)a);
            }
        }
    }
    for (int n = 0; n < headn; ++n) {
        double b = (double)f.b(nh)[n];
        for (int k = 0; k < mid; ++k) b += (double)f.w(nh)[n * mid + k] * (double)f.b(n2)[k];
        o[C::OFF_B + n] = (float)b;
    }
    return off;
}

// weight slots of upcat_tc_kernel in its step order: A(half 0) x 6 | 9 skip chunks | 3 up chunks | A(half 1) x 6 | 3 up chunks
int64_t pack_upcat_tc(std::vector<float>& out, const Folded& f) {
    using C = CfgUpCatTc;
    pad4(out);
    while (out.size() % 32) out.push_back(0.f);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    const float* w = f.w("conv4_1_1");    // [96][232]
    const float* wt = f.w("deconv5_1");   // [cin 96][cout 96][2][2]
    int slot = 0;
    auto a_steps = [&](int h) {
        for (int kc = 0; kc < C::NKA; ++kc, ++slot) {
            float* sb = o + (int64_t)slot * C::SLOT;
            for (int par = 0; par < 4; ++par)
                for (int ml = 0; ml < 48; ++ml)
                    for (int kl = 0; kl < C::MC; ++kl) {
                        const int c = kc * C::MC + kl, m = 48 * h + ml;
                        put_kmajor_split(sb, sb + C::NHALF * C::MC, par * 48 + ml, kl, C::MC, wt[((c * 96 + m) * 2 + (par >> 1)) * 2 + (par & 1)]);
                    }
        }
    };
    auto b_step = [&](int k0, int kvalid) {      // concat rows [k0, k0 + 16), the first kvalid of them real
        float* sb = o + (int64_t)slot * C::SLOT;
        for (int n = 0; n < C::N; ++n)
            for (int kl = 0; kl < kvalid; ++kl) put_kmajor_split(sb, sb + C::N * C::MC, n, kl, C::MC, w[n * 232 + k0 + kl]);
        ++slot;
    };
    a_steps(0);
    for (int c = 0; c < C::NSKIP; ++c) b_step(c * C::MC, std::min(C::MC, C::CS - c * C::MC));
    for (int j = 0; j < C::NUPH; ++j) b_step(C::CS + j * C::MC, C::MC);
    a_steps(1);
    for (int j = 0; j < C::NUPH; ++j) b_step(C::CS + 48 + j * C::MC, C::MC);
    for (int m = 0; m < 96; ++m) o[C::OFF_BT + m] = f.b("deconv5_1")[m];
    for (int n = 0; n < 96; ++n) o[C::OFF_B + n] = f.b("conv4_1_1")[n];
    return off;
}

// weight slots of irbtc2_kernel in its step order: per half { CIN/16 expand K chunks | CMID/NH/16 mid chunks }
template <class C>
int64_t pack_irbtc2(std::vector<float>& out, const Folded& f, const std::string& n1, const std::string& nd, const std::string& n2) {
    pad4(out);
    while (out.size() % 32) out.push_back(0.f);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    int slot = 0;
    for (int h = 0; h < C::NH; ++h) {
        for (int kc = 0; kc < C::NKA; ++kc, ++slot) {
            float* sb = o + (int64_t)slot * C::SLOT;
            for (int ml = 0; ml < C::NA; ++ml) {
                const int m = h * C::NA + ml;
                if (m >= C::CMID) continue;
                for (int kl = 0; kl < C::MC; ++kl) put_kmajor_split(sb, sb + C::NA * C::MC, ml, kl, C::MC, f.w(n1)[m * C::CIN + kc * C::MC + kl]);
            }
        }
        for (int j = 0; j < C::NMC; ++j, ++slot) {
            float* sb = o + (int64_t)slot * C::SLOT;
            for (int ml = 0; ml < C::MC; ++ml) {
                const int m = h * C::NA + j * C::MC + ml;
                if (m >= C::CMID) continue;
                sb[C::OFF_B1 + ml] = f.b(n1)[m];
                for (int t = 0; t < 9; ++t) sb[C::OFF_WD + ml * 9 + t] = f.w(nd)[m * 9 + t];
                sb[C::OFF_BD + ml] = f.b(nd)[m];
                for (int n = 0; n < C::COUT; ++n) put_kmajor_split(sb + C::OFF_W2, sb + C::OFF_W2 + C::COUTP * C::MC, n, ml, C::MC, f.w(n2)[n * C::CMID + m]);
            }
        }
    }
    for (int n = 0; n < C::COUT; ++n) o[C::OFF_B2 + n] = f.b(n2)[n];
    return off;
}

template <class C>
int64_t pack_dwpwtc(std::vector<float>& out, const Folded& f, const std::string& nd, const std::string& n2) {
    pad4(out);
    while (out.size() % 32) out.push_back(0.f);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    for (int c = 0; c < C::NCHUNK; ++c) {
        float* cb = o + (int64_t)c * C::CB;
        for (int ml = 0; ml < C::MC; ++ml) {
            const int m = c * C::MC + ml;
            for (int t = 0; t < C::KK; ++t) cb[C::OFF_WD + ml * C::KK + t] = f.w(nd)[m * C::KK + t];
            cb[C::OFF_BD + ml] = f.b(nd)[m];
            for (int n = 0; n < C::N; ++n) put_kmajor_split(cb + C::OFF_WH, cb + C::OFF_WL, n, ml, C::MC, f.w(n2)[n * C::C + m]);
        }
    }
    for (int n = 0; n < C::N; ++n) o[C::OFF_B + n] = f.b(n2)[n];
    return off;
}

template <class C>
int64_t pack_irbtc(std::vector<float>& out, const Folded& f, const std::string& n1, const std::string& nd, const std::string& n2) {
    pad4(out);
    while (out.size() % 32) out.push_back(0.f);          // bulk copies and UMMA descriptors want 128-byte aligned blocks
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    for (int c = 0; c < C::NCHUNK; ++c) {
        float* cb = o + C::OFF_CH + (int64_t)c * C::CB;
        for (int ml = 0; ml < C::MC; ++ml) {
            const int m = c * C::MC + ml;
            if (m >= C::CMID) continue;                      // zero padding of the mid channels
            // expand weights: one resident B operand over all mid channels (E1ALL), or one per chunk block
            for (int k = 0; k < C::CIN; ++k) {
                if (C::E1ALL) put_kmajor_split(o + C::OFF_W1H, o + C::OFF_W1L, m, k, C::CIN, f.w(n1)[m * C::CIN + k]);
                else put_kmajor_split(cb + C::OFF_W1H, cb + C::OFF_W1L, ml, k, C::CIN, f.w(n1)[m * C::CIN + k]);
            }
            cb[C::OFF_B1 + ml] = f.b(n1)[m];
            for (int t = 0; t < 9; ++t) cb[C::OFF_WD + ml * 9 + t] = f.w(nd)[m * 9 + t];
            cb[C::OFF_BD + ml] = f.b(nd)[m];
            // project weights as one B operand of 2*COUTP rows: rows [0, COUTP) = hi parts, rows [COUTP, 2*COUTP) = lo parts
            for (int n = 0; n < C::COUT; ++n)
                put_kmajor_split(cb + C::OFF_W2, cb + C::OFF_W2 + C::COUTP * C::MC, n, ml, C::MC, f.w(n2)[n * C::CMID + m]);
        }
    }
    for (int n = 0; n < C::COUT; ++n) o[C::OFF_B2 + n] = f.b(n2)[n];
    return off;
}

// channel-lane tensor-core block (yf_tct.cuh):
// [W1hi: 128 x KX][W1lo][W2: (hi | lo) x CMID][wd: CMID x 9][bd][b2]; column CIN of W1 is the expand bias (the ones channel)
template <class C>
int64_t pack_irbt(std::vector<float>& out, const Folded& f, const std::string& n1, const std::string& nd, const std::string& n2) {
    pad4(out);
    while (out.size() % 32) out.push_back(0.f);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    for (int m = 0; m < C::CMID; ++m) {
        for (int k = 0; k < C::CIN; ++k) put_kmajor_split(o + C::OFF_W1H, o + C::OFF_W1L, m, k, C::KX, f.w(n1)[m * C::CIN + k]);
        put_kmajor_split(o + C::OFF_W1H, o + C::OFF_W1L, m, C::CIN, C::KX, f.b(n1)[m]);
        for (int t = 0; t < 9; ++t) o[C::OFF_WD + m * 9 + t] = f.w(nd)[m * 9 + t];
        o[C::OFF_BD + m] = f.b(nd)[m];
        for (int n = 0; n < C::COUT; ++n)
            put_kmajor_split(o + C::OFF_W2, o + C::OFF_W2 + C::COUTP * C::CMID, n, m, C::CMID, f.w(n2)[n * C::CMID + m]);
    }
    for (int n = 0; n < C::COUT; ++n) o[C::OFF_B2 + n] = f.b(n2)[n];
    return off;
}

// stem on the warp-streaming engine: [W0: 9 x 8][b0][W1: 8 x 8 (k-major)][b1][Wd: 9 x 8][bd][W2: 4 x 8 (n-major)][b2]
template <class C>
int64_t pack_wstem(std::vector<float>& out, const Folded& f) {
    pad4(out);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    for (int c = 0; c < 8; ++c) {
        for (int t = 0; t < 9; ++t) o[C::OFF_W0 + t * 8 + c] = f.w("conv0")[c * 9 + t];
        o[C::OFF_B0 + c] = f.b("conv0")[c];
        for (int k = 0; k < 8; ++k) o[C::OFF_W1 + k * 8 + c] = f.w("conv1_2")[c * 8 + k];
        o[C::OFF_B1 + c] = f.b("conv1_2")[c];
        for (int t = 0; t < 9; ++t) o[C::OFF_WD + t * 8 + c] = f.w("conv1_3")[c * 9 + t];
        o[C::OFF_BD + c] = f.b("conv1_3")[c];
        for (int n = 0; n < 4; ++n) o[C::OFF_W2 + n * 8 + c] = f.w("conv1_4")[n * 8 + c];
    }
    for (int n = 0; n < 4; ++n) o[C::OFF_B2 + n] = f.b("conv1_4")[n];
    return off;
}

template <class C>
int64_t pack_stem(std::vector<float>& out, const Folded& f) {
    pad4(out);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    for (int c = 0; c < 8; ++c)                          // conv0 weight [8][CIN][3][3] -> [ci][tap][c]
        for (int ci = 0; ci < C::CIN; ++ci)
            for (int t = 0; t < 9; ++t) o[C::OFF_W0 + (ci * 9 + t) * 8 + c] = f.w("conv0")[(c * C::CIN + ci) * 9 + t];
    for (int c = 0; c < 8; ++c) o[C::OFF_B0 + c] = f.b("conv0")[c];
    for (int m = 0; m < 8; ++m)
        for (int k = 0; k < 8; ++k) o[C::OFF_W1 + k * 8 + m] = f.w("conv1_2")[m * 8 + k];
    for (int m = 0; m < 8; ++m) o[C::OFF_B1 + m] = f.b("conv1_2")[m];
    for (int i = 0; i < 72; ++i) o[C::OFF_WD + i] = f.w("conv1_3")[i];
    for (int m = 0; m < 8; ++m) o[C::OFF_BD + m] = f.b("conv1_3")[m];
    for (int n = 0; n < 4; ++n)
        for (int m = 0; m < 8; ++m) o[C::OFF_W2 + m * 4 + n] = f.w("conv1_4")[n * 8 + m];
    for (int n = 0; n < 4; ++n) o[C::OFF_B2 + n] = f.b("conv1_4")[n];
    return off;
}

// dense_tc_kernel: 27 resident B operands (channel block cb, tap t): 64 rows x 8 input channels, rows 0..23 = hi, 24..47 = lo of W9
int64_t pack_dense_tc(std::vector<float>& out, const Folded& f) {
    using C = CfgDenseTc;
    pad4(out);
    while (out.size() % 32) out.push_back(0.f);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    const float* w9 = f.w("conv1_9");   // [24][24][3][3]
    for (int cb = 0; cb < 3; ++cb)
        for (int t = 0; t < 9; ++t) {
            float* blk = o + (int64_t)(cb * 9 + t) * 512;
            for (int n = 0; n < 24; ++n)
                for (int kl = 0; kl < 8; ++kl) put_kmajor_split(blk, blk + 24 * 8, n, kl, 8, w9[((n * 24 + cb * 8 + kl) * 3 + t / 3) * 3 + t % 3]);
        }
    for (int c = 0; c < 24; ++c)                                                // [24][4] -> [c / 4][k][c % 4]: one 128-bit load = 4 channels of one k
        for (int k = 0; k < 4; ++k) o[C::OFF_W8 + (c / 4) * 16 + k * 4 + (c % 4)] = f.w("conv1_8")[c * 4 + k];
    for (int i = 0; i < 24; ++i) { o[C::OFF_B8 + i] = f.b("conv1_8")[i]; o[C::OFF_B9 + i] = f.b("conv1_9")[i]; }
    for (int j = 0; j < 8; ++j)
        for (int n = 0; n < 24; ++n) o[C::OFF_W21 + n * 8 + j] = f.w("conv2_1")[j * 24 + n];        // [8][24] -> transposed [24][8]
    for (int i = 0; i < 8; ++i) o[C::OFF_B21 + i] = f.b("conv2_1")[i];
    return off;
}

int64_t pack_dense(std::vector<float>& out, const Folded& f) {
    using C = CfgDense;
    pad4(out);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    const float* w8 = f.w("conv1_8");   // [24][4]
    const float* w9 = f.w("conv1_9");   // [24][24][3][3]
    for (int c = 0; c < C::NCHUNK; ++c) {
        float* cb = o + (int64_t)c * C::CB;
        for (int ml = 0; ml < C::MC; ++ml) {
            const int m = c * C::MC + ml;
            for (int k = 0; k < 4; ++k) cb[C::OFF_W1 + k * C::MC + ml] = w8[m * 4 + k];
            cb[C::OFF_B1 + ml] = f.b("conv1_8")[m];
            for (int dy = 0; dy < 3; ++dy)
                for (int cg = 0; cg < 3; ++cg)
                    for (int dx = 0; dx < 3; ++dx)
                        for (int n = 0; n < 8; ++n)
                            cb[C::OFF_WC + ((ml * 3 + dy) * 3 + cg) * 24 + dx * 8 + n] = w9[(((cg * 8 + n) * 24 + m) * 3 + dy) * 3 + dx];
        }
    }
    for (int n = 0; n < 24; ++n) o[C::OFF_B9 + n] = f.b("conv1_9")[n];
    for (int n = 0; n < 8; ++n)
        for (int m = 0; m < 24; ++m) o[C::OFF_W3 + m * 8 + n] = f.w("conv2_1")[n * 24 + m];
    for (int n = 0; n < 8; ++n) o[C::OFF_B3 + n] = f.b("conv2_1")[n];
    return off;
}

int64_t pack_lite34(std::vector<float>& out, const Folded& f) {
    using C = CfgLite34;
    pad4(out);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    for (int m = 0; m < C::M; ++m) {
        for (int k = 0; k < C::K; ++k) o[C::OFF_W1 + k * C::M + m] = f.w("conv3_2")[m * C::K + k];
        o[C::OFF_B1 + m] = f.b("conv3_2")[m];
        for (int n = 0; n < C::N; ++n) o[C::OFF_W2 + m * C::N + n] = f.w("conv3_4")[n * C::M + m];
    }
    for (int n = 0; n < C::N; ++n) o[C::OFF_B2 + n] = f.b("conv3_4")[n];
    return off;
}

int64_t pack_pw52(std::vector<float>& out, const Folded& f) {
    using C = CfgPw52;
    pad4(out);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    for (int n = 0; n < C::N; ++n)
        for (int k = 0; k < C::K; ++k) o[k * C::N + n] = f.w("conv5_2")[n * C::K + k];
    for (int n = 0; n < C::N; ++n) o[C::K * C::N + n] = f.b("conv5_2")[n];
    return off;
}

int64_t pack_upcat(std::vector<float>& out, const Folded& f) {
    using C = CfgUpCat;
    pad4(out);
    const int64_t off = (int64_t)out.size();
    out.resize(off + C::WFLOATS, 0.f);
    float* o = out.data() + off;
    const float* w = f.w("conv4_1_1");    // [96][232]
    for (int n = 0; n < 96; ++n) {
        for (int k = 0; k < 136; ++k) o[C::OFF_WAB + k * 96 + n] = w[n * 232 + k];                    // rows 136..CSP-1 stay zero
        for (int k = 0; k < 96; ++k) o[C::OFF_WAB + (C::CSP + k) * 96 + n] = w[n * 232 + 136 + k];
        o[C::OFF_B + n] = f.b("conv4_1_1")[n];
    }
    const float* wt = f.w("deconv5_1");   // [cin 96][cout 96][2][2]
    for (int c = 0; c < 96; ++c)
        for (int py = 0; py < 2; ++py)
            for (int px = 0; px < 2; ++px)
                for (int m = 0; m < 96; ++m)
                    o[C::OFF_WT + ((c * 4) + py * 2 + px) * 96 + m] = wt[((c * 96 + m) * 2 + py) * 2 + px];
    for (int m = 0; m < 96; ++m) o[C::OFF_BT + m] = f.b("deconv5_1")[m];
    return off;
}

template <class C>
Group make_wirb(const char* name, int out_ch) {
    Group g{};
    g.name = name;
    g.launch = &launch_wirb<C>;
    g.out_ch = out_ch;
    return g;
}

template <class C>
Group make_dwpwtc(const char* name, int out_ch) {
    Group g{};
    g.name = name;
    g.launch = &launch_dwpwtc<C>;
    g.occupancy = &occ_dwpwtc<C>;
    g.out_ch = out_ch;
    return g;
}

template <class C>
Group make_irbtc2(const char* name, int out_ch) {
    Group g{};
    g.name = name;
    g.launch = &launch_irbtc2<C>;
    g.occupancy = &occ_irbtc2<C>;
    g.out_ch = out_ch;
    return g;
}

template <class C>
Group make_irbtc(const char* name, int out_ch) {
    Group g{};
    g.name = name;
    g.launch = &launch_irbtc<C>;
    g.occupancy = &occ_irbtc<C>;
    g.out_ch = out_ch;
    return g;
}

template <class C>
Group make_irb(const char* name, int out_ch) {
    Group g{};
    g.name = name;
    g.launch = &launch_irb<C>;
    g.occupancy = &occ_irb<C>;
    g.out_ch = out_ch;
    return g;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// lifecycle
// ---------------------------------------------------------------------------------------------
extern "C" int yf_abi_version(void) { return YF_ABI_VERSION; }

extern "C" const char* yf_last_error(const yf_ctx* ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }

extern "C" int64_t yf_weight_count_variant(int in_ch, int num_cls, int num_anchors, int variant) {
    if (in_ch < 1 || num_cls < 1 || num_anchors < 1 || (variant != YF_VARIANT_FULL && variant != YF_VARIANT_LITE)) return -1;
    return build_specs(in_ch, num_cls, num_anchors, variant).total;
}
extern "C" int64_t yf_weight_count(int in_ch, int num_cls, int num_anchors) { return yf_weight_count_variant(in_ch, num_cls, num_anchors, YF_VARIANT_FULL); }

// Post-processing workspace: everything a ctx needs for yf_postprocess / yf_decode / yf_val_nms / yf_nms_sorted_*. Allocated at
// creation; the forward's activation, head and staging buffers (2 GB at 640x512, batch 256) come with the first yf_load_weights, so
// a context that only ever post-processes (YOLO_post_process, val.non_max_suppression) stays small.
static int alloc_post(yf_ctx* ctx) {
    const int B = ctx->max_batch, H = ctx->H, W = ctx->W;
    CU(cudaMalloc(&ctx->d_counts, sizeof(int32_t) * B));
    CU(cudaMalloc(&ctx->d_status, sizeof(int32_t) * B));
    ctx->NC = ctx->num_anchors * ((H / 16) * (W / 16) + (H / 32) * (W / 32));
    const size_t n = (size_t)ctx->NC * B;
    CU(cudaMalloc(&ctx->p_rec, sizeof(yf_det) * n));
    CU(cudaMalloc(&ctx->p_conf, sizeof(double) * n));
    CU(cudaMalloc(&ctx->p_cls, sizeof(int32_t) * n));
    CU(cudaMalloc(&ctx->p_sbox, sizeof(int4) * n));
    CU(cudaMalloc(&ctx->p_order, sizeof(int32_t) * n));
    CU(cudaMalloc(&ctx->p_alive, n));
    return YF_OK;
}

static int alloc_forward(yf_ctx* ctx) {
    if (!ctx->d_act.empty()) return YF_OK;
    const int B = ctx->max_batch, H = ctx->H, W = ctx->W;
    auto dim = [&](int div, int& h, int& w) { h = H / div; w = W / div; };
    // (name, channels, divisor) of every group output, in launch order
    struct Out { const char* name; int ch; int div; };
    const Out outs[] = {
        {"conv1_4", 4, 2}, {"res1_1", 4, 2}, {"conv2_1", 8, 4}, {"res2_1", 8, 4}, {"res2_2", 8, 4}, {"conv3_1", 8, 8},
        {"res3_1", 8, 8}, {"res3_2", 8, 8}, {"conv3_4", 16, 8}, {"res3_3", 16, 8}, {"res3_4", 16, 8}, {"res3_5", 16, 8},
        {"res3_6", 16, 8}, {"conv4_1", 24, 16}, {"res4_1", 24, 16}, {"res4_2", 24, 16}, {"res4_3", 24, 16}, {"res4_4", 24, 16},
        {"conv5_1", 48, 32}, {"res5_1", 48, 32}, {"res5_2", 48, 32}, {"res5_3", 48, 32}, {"res5_4", 48, 32}, {"res5_5", 48, 32},
        {"conv5_2", 96, 32}, {"conv5_4", 128, 32}, {"conv4_1_1", 96, 16}, {"conv4_1_3", 96, 16}};
    for (const Out& o : outs) {
        int h, w;
        dim(o.div, h, w);
        const int64_t per = (int64_t)o.ch * h * w;
        float* p = nullptr;
        CU(cudaMalloc(&p, sizeof(float) * per * B));
        ctx->d_act.push_back(p);
        ctx->taps[o.name] = {p, per};
    }
    {
        const int64_t per = (int64_t)136 * (H / 16) * (W / 16);
        CU(cudaMalloc(&ctx->d_skip, sizeof(float) * per * B));
        ctx->taps["conv4_2"] = {ctx->d_skip, per};
    }
    const int64_t hl = (int64_t)ctx->nout * (H / 16) * (W / 16), hs = (int64_t)ctx->nout * (H / 32) * (W / 32);
    CU(cudaMalloc(&ctx->d_hl, sizeof(float) * hl * B));
    CU(cudaMalloc(&ctx->d_hs, sizeof(float) * hs * B));
    CU(cudaMalloc(&ctx->d_x, sizeof(float) * (int64_t)ctx->in_ch * H * W * B));
    CU(cudaMalloc(&ctx->d_u8, (size_t)ctx->in_ch * H * W * B));
    return YF_OK;
}

static int ensure_out(yf_ctx* ctx, int max_det) {
    if (max_det <= ctx->out_cap) return YF_OK;
    for (auto& kv : ctx->graphs) cudaGraphExecDestroy(kv.second.first);      // graphs bake the output pointer in
    ctx->graphs.clear();
    if (ctx->d_out) CU(cudaFree(ctx->d_out));
    ctx->d_out = nullptr;
    CU(cudaMalloc(&ctx->d_out, sizeof(yf_det) * (size_t)max_det * ctx->max_batch));
    ctx->out_cap = max_det;
    return YF_OK;
}

static void build_plan(yf_ctx* ctx) {
    const int H = ctx->H, W = ctx->W;
    std::vector<Group>& G = ctx->groups;
    G.clear();
    int ai = 0;   // index into d_act
    auto hw = [&](Group& g, int din, int dout) {
        g.a.Hin = H / din; g.a.Win = W / din; g.a.Hout = H / dout; g.a.Wout = W / dout;
    };
    const float* prev = nullptr;
    auto chain = [&](Group g, int din, int dout) {
        hw(g, din, dout);
        g.a.x = prev;
        g.a.y = ctx->d_act[ai++];
        prev = g.a.y;
        G.push_back(g);
    };
    {
        Group g{}; g.name = "conv1_4"; g.out_ch = 4;
        if (ctx->in_ch == 3) { g.launch = &launch_stem<CfgStem3>; g.occupancy = &occ_stem3; }
        else if (YF_USE_WIRB) { g.launch = &launch_wstem<CfgStemW>; }
        else { g.launch = &launch_stem<CfgStem>; g.occupancy = &occ_stem; }
        g.a.Hin = H; g.a.Win = W; g.a.Hout = H / 2; g.a.Wout = W / 2;
        g.a.y = ctx->d_act[ai++]; prev = g.a.y; G.push_back(g);
    }
#if YF_USE_WIRB
    chain(make_wirb<CfgRes1W>("res1_1", 4), 2, 2);
#else
    chain(make_irb<CfgRes1>("res1_1", 4), 2, 2);
#endif
#if YF_DENSE_TC
    {
        Group g{}; g.name = "conv2_1"; g.launch = &launch_dense_tc; g.occupancy = &occ_dense_tc; g.out_ch = 8;
        if (YF_DENSE_TA) { g.launch = &launch_dense_ta; g.occupancy = &occ_dense_ta; g.a.small = &ctx->dense_small; }
        chain(g, 2, 4);
    }
#else
    { Group g{}; g.name = "conv2_1"; g.launch = &launch_dense; g.occupancy = &occ_dense; g.out_ch = 8; chain(g, 2, 4); }
#endif
#if YF_USE_WIRB
    chain(make_wirb<CfgRes2W>("res2_1", 8), 4, 4);
    chain(make_wirb<CfgRes2W>("res2_2", 8), 4, 4);
    chain(make_wirb<CfgDown2W>("conv3_1", 8), 4, 8);
#else
    chain(make_irb<CfgRes2>("res2_1", 8), 4, 4);
    chain(make_irb<CfgRes2>("res2_2", 8), 4, 4);
    chain(make_irb<CfgDown2>("conv3_1", 8), 4, 8);
#endif
    for (const char* n : {"res3_1", "res3_2"}) {
        Group g = make_irb<CfgRes3a>(n, 8);
        if (YF_USE_TC && YF_USE_TCT_A) { g.launch = &launch_irbt0<CfgRes3aTt>; g.occupancy = &occ_irbt<CfgRes3aTt>; }
        chain(g, 8, 8);
    }
    if (ctx->variant == YF_VARIANT_LITE) { Group g{}; g.name = "conv3_4"; g.launch = &launch_lite34; g.out_ch = 16; chain(g, 8, 8); }
    else {
        Group g = make_irb<CfgWide3>("conv3_4", 16);
        if (YF_USE_TC && YF_USE_TCT_A) { g.launch = &launch_irbt0<CfgWide3Tt>; g.occupancy = &occ_irbt<CfgWide3Tt>; }
        chain(g, 8, 8);
    }
#if YF_USE_TC
    for (const char* n : {"res3_3", "res3_4", "res3_5", "res3_6"}) {
        Group g = make_irbtc<CfgRes3bTc>(n, 16);
#if YF_USE_TCT
        g.launch = &launch_irbt0<CfgRes3bTt>; g.occupancy = &occ_irbt<CfgRes3bTt>;
#else
        g.launch = &launch_irbtc_auto<CfgRes3bTc, CfgRes3bTcS, CfgRes3bTcXS>;
#endif
        chain(g, 8, 8);
    }
#else
    chain(make_irb<CfgRes3b>("res3_3", 16), 8, 8);
    chain(make_irb<CfgRes3b>("res3_4", 16), 8, 8);
    chain(make_irb<CfgRes3b>("res3_5", 16), 8, 8);
    chain(make_irb<CfgRes3b>("res3_6", 16), 8, 8);
#endif
    {
        Group g = make_irb<CfgDown3>("conv4_1", 24);
        g.launch = &launch_irb_auto<CfgDown3, CfgDown3N>;
        if (YF_USE_TC && YF_USE_TCT_A) { g.launch = &launch_irbt0<CfgDown3Tt>; g.occupancy = &occ_irbt<CfgDown3Tt>; }
        chain(g, 8, 16);
    }
#if YF_USE_TC
    for (const char* n : {"res4_1", "res4_2", "res4_3", "res4_4"}) {
        Group g = make_irbtc<CfgRes4Tc>(n, 24);
#if YF_USE_TCT
        g.launch = &launch_res4_auto<CfgRes4Tt, CfgRes4Tc, CfgRes4TcS, CfgRes4TcXS>;
#else
        g.launch = &launch_irbtc_auto<CfgRes4Tc, CfgRes4TcS, CfgRes4TcXS>;
#endif
        chain(g, 16, 16);
    }
#else
    chain(make_irb<CfgRes4>("res4_1", 24), 16, 16);
    chain(make_irb<CfgRes4>("res4_2", 24), 16, 16);
    chain(make_irb<CfgRes4>("res4_3", 24), 16, 16);
    chain(make_irb<CfgRes4>("res4_4", 24), 16, 16);
#endif
    {
        Group g = make_irb<CfgDown4>("conv5_1", 48);
        g.launch = &launch_irb_auto<CfgDown4, CfgDown4N>;
        if (YF_USE_TC && YF_USE_TCT_A) g.launch = &launch_down4_auto<CfgDown4Tt, CfgDown4, CfgDown4N>;
        g.a.skip = ctx->d_skip;
        chain(g, 16, 32);
    }
#if YF_RES5_TC
    for (const char* n : {"res5_1", "res5_2", "res5_3", "res5_4", "res5_5"}) {
        Group g = make_irbtc2<CfgRes5Tc>(n, 48);
        g.launch = &launch_irbtc2_auto<CfgRes5Tc, CfgRes5TcS>;
        chain(g, 32, 32);
    }
#else
    for (const char* n : {"res5_1", "res5_2", "res5_3", "res5_4", "res5_5"}) chain(make_irb<CfgRes5>(n, 48), 32, 32);
#endif
    { Group g{}; g.name = "conv5_2"; g.launch = &launch_pw52; g.out_ch = 96; chain(g, 32, 32); }
    const float* conv5_2 = prev;
#if YF_USE_TC
    { Group g = make_dwpwtc<CfgNeckS1Tc>("conv5_4", 128); g.launch = &launch_dwpwtc_auto<CfgNeckS1Tc, CfgNeckS1TcS, CfgNeckS1TcN>; chain(g, 32, 32); }
#else
    chain(make_irb<CfgNeckS1>("conv5_4", 128), 32, 32);
#endif
    {
        Group g = heads_on_tc(ctx->nout) ? make_dwpwtc<CfgNeckS2Tc>("head_5", 0) : make_irb<CfgNeckS2>("head_5", 0);   // y = caller's head_small, set per call
        if (heads_on_tc(ctx->nout)) g.launch = &launch_dwpwtc_auto<CfgNeckS2Tc, CfgNeckS2TcS, CfgNeckS2TcN>;
        hw(g, 32, 32); g.a.x = prev; g.a.headn = ctx->nout; G.push_back(g);
    }
    if (ctx->variant == YF_VARIANT_LITE) return;        // the lite forward ends at head_5 (yolo_fastest.py:365-372)
    {
        Group g{}; g.name = "conv4_1_1"; g.out_ch = 96;
        if (upcat_on_tc(ctx->H, ctx->W)) { g.launch = &launch_upcat_tc; g.occupancy = &occ_upcat_tc; }
        else { g.launch = &launch_upcat; g.occupancy = &occ_upcat; }
        hw(g, 16, 16); g.a.x = ctx->d_skip; g.a.x2 = conv5_2; g.a.y = ctx->d_act[ai++]; prev = g.a.y; G.push_back(g);
    }
#if YF_USE_TC
    { Group g = make_dwpwtc<CfgNeckL1Tc>("conv4_1_3", 96); g.launch = &launch_dwpwtc_auto<CfgNeckL1Tc, CfgNeckL1TcS, CfgNeckL1TcN>; chain(g, 16, 16); }
#else
    chain(make_irb<CfgNeckL1>("conv4_1_3", 96), 16, 16);
#endif
    {
        Group g = heads_on_tc(ctx->nout) ? make_dwpwtc<CfgNeckL2Tc>("head_4", 0) : make_irb<CfgNeckL2>("head_4", 0);   // y = caller's head_large
        if (heads_on_tc(ctx->nout)) g.launch = &launch_dwpwtc_auto<CfgNeckL2Tc, CfgNeckL2TcS, CfgNeckL2TcN>;
        hw(g, 16, 16); g.a.x = prev; g.a.headn = ctx->nout; G.push_back(g);
    }
}

static void set_sm_count(yf_ctx* ctx) {
    int nsm = 148;
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, ctx->device);
    for (Group& g : ctx->groups) {
        g.a.nsm = nsm;
        g.a.resident = nsm * (g.occupancy ? g.occupancy() : 1);
        g.a.tc = &g.tcache;              // the plan is complete: group addresses are stable from here on
    }
}

extern "C" int yf_create(yf_ctx** out, int device, int in_ch, int num_cls, int num_anchors, int max_batch, int H, int W) {
    return yf_create_variant(out, device, in_ch, num_cls, num_anchors, max_batch, H, W, YF_VARIANT_FULL);
}

extern "C" int yf_create_variant(yf_ctx** out, int device, int in_ch, int num_cls, int num_anchors, int max_batch, int H, int W, int variant) {
    if (!out) { set_err(nullptr, "out is null"); return YF_ERR_ARG; }
    *out = nullptr;
    if (variant != YF_VARIANT_FULL && variant != YF_VARIANT_LITE) { set_err(nullptr, "unknown model variant %d", variant); return YF_ERR_ARG; }
    if (variant == YF_VARIANT_LITE && in_ch != 1) { set_err(nullptr, "YoloFastest_lite is served for single-channel input"); return YF_ERR_ARG; }
    if (in_ch != 1 && in_ch != 3) { set_err(nullptr, "in_ch=%d unsupported: 1 (the shipped models, _config.py:10) or 3 (colour input)", in_ch); return YF_ERR_ARG; }
    if (num_cls < 1 || num_cls > POST_MAX_CLS || num_anchors < 1 || num_anchors > YF_MAX_ANCHORS || max_batch < 1) {
        set_err(nullptr, "bad num_cls/num_anchors/max_batch (%d, %d, %d)", num_cls, num_anchors, max_batch);
        return YF_ERR_ARG;
    }
    if (H < 32 || W < 32 || H % 32 || W % 32) { set_err(nullptr, "H, W must be positive multiples of 32 (got %dx%d)", H, W); return YF_ERR_ARG; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || device < 0 || device >= ndev) {
        set_err(nullptr, "no usable CUDA device %d (%s); this library has no CPU fallback", device,
                e != cudaSuccess ? cudaGetErrorString(e) : "index out of range");
        return YF_ERR_CUDA;
    }
    yf_ctx* ctx = new yf_ctx();
    ctx->device = device; ctx->in_ch = in_ch; ctx->num_cls = num_cls; ctx->num_anchors = num_anchors;
    ctx->max_batch = max_batch; ctx->H = H; ctx->W = W; ctx->variant = variant;
    ctx->nout = head_channels(num_cls, num_anchors, variant);
    ctx->specs = build_specs(in_ch, num_cls, num_anchors, variant);
    auto fail = [&](int rc) { g_err = ctx->err; yf_destroy(ctx); return rc; };
    if ((e = cudaSetDevice(device)) != cudaSuccess) { set_err(&ctx->err, "cudaSetDevice: %s", cudaGetErrorString(e)); return fail(YF_ERR_CUDA); }
    cudaError_t ie[] = {
        cudaFuncSetAttribute(stem_kernel<CfgStem, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgStem::SMEM_BYTES),
        cudaFuncSetAttribute(stem_kernel<CfgStem, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgStem::SMEM_BYTES),
        cudaFuncSetAttribute(stem_kernel<CfgStem3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgStem3::SMEM_BYTES),
        cudaFuncSetAttribute(stem_kernel<CfgStem3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgStem3::SMEM_BYTES),
        cudaFuncSetAttribute(dense_kernel<CfgDense>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgDense::SMEM_BYTES),
        cudaFuncSetAttribute(dense_tc_kernel<CfgDenseTc>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgDenseTc::SMEM_BYTES),
        cudaFuncSetAttribute(dense_ta_kernel<DenseTaCfg>, cudaFuncAttributeMaxDynamicSharedMemorySize, DenseTaCfg::SMEM_BYTES),
        cudaFuncSetAttribute(pw_kernel<CfgPw52>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgPw52::SMEM_BYTES),
        cudaFuncSetAttribute(upcat_kernel<CfgUpCat>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgUpCat::SMEM_BYTES),
        cudaFuncSetAttribute(upcat_tc_kernel<CfgUpCatTc>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgUpCatTc::SMEM_BYTES),
        init_irb<CfgRes1>(),
        init_wirb<CfgRes1W>(), init_wirb<CfgRes2W>(), init_wirb<CfgDown2W>(), init_wstem<CfgStemW>(),
        cudaFuncSetAttribute(post_kernel<YF_MODE_DETECT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 * 12),
        cudaFuncSetAttribute(post_kernel<YF_MODE_VALIDATE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 * 12),
        cudaFuncSetAttribute(post_kernel<POST_SRC_ROWS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 * 12),
        cudaFuncSetAttribute(prep_frames_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PREP_SMEM_CAP),
        cudaFuncSetAttribute(prep_frames_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, PREP_SMEM_CAP),
        cudaFuncSetAttribute(jpeg_entropy_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, JPEG_TABS_BYTES),
        cudaFuncSetAttribute(jpeg_entropy_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * JPEG_TABS_BYTES),
        init_irb<CfgRes2>(), init_irb<CfgDown2>(), init_irb<CfgRes3a>(), init_irb<CfgWide3>(),
        init_irb<CfgRes3b>(), init_irbtc<CfgRes3bTc>(), init_irbt<CfgRes3bTt>(), init_irbt<CfgRes4Tt>(), init_irbt<CfgRes3aTt>(), init_irbt<CfgWide3Tt>(), init_irbt<CfgDown3Tt>(), init_irbt<CfgDown4Tt>(), init_irbtc<CfgRes4Tc>(), init_irbtc2<CfgRes5Tc>(), init_irbtc2<CfgRes5TcS>(), init_irbtc2<CfgRes5TcXS>(), init_irbtc2<CfgRes5TcN>(), init_dwpwtc<CfgNeckS1TcS>(), init_dwpwtc<CfgNeckS2TcS>(), init_irbtc<CfgRes3bTcXS>(), init_irbtc<CfgRes4TcXS>(), init_dwpwtc<CfgNeckS1TcN>(), init_dwpwtc<CfgNeckS2TcN>(), init_dwpwtc<CfgNeckL1TcN>(), init_dwpwtc<CfgNeckL2TcN>(), init_irb<CfgDown3N>(), init_irb<CfgDown4N>(), init_dwpwtc<CfgNeckL1TcS>(), init_dwpwtc<CfgNeckL2TcS>(), init_irbtc<CfgRes3bTcS>(), init_irbtc<CfgRes4TcS>(), init_dwpwtc<CfgNeckS1Tc>(), init_dwpwtc<CfgNeckL1Tc>(), init_dwpwtc<CfgNeckS2Tc>(), init_dwpwtc<CfgNeckL2Tc>(), init_irb<CfgDown3>(), init_irb<CfgRes4>(), init_irb<CfgDown4>(), init_irb<CfgRes5>(),
        init_irb<CfgNeckS1>(), init_irb<CfgNeckS2>(), init_irb<CfgNeckL1>(), init_irb<CfgNeckL2>()};
    for (cudaError_t x : ie)
        if (x != cudaSuccess) { set_err(&ctx->err, "cudaFuncSetAttribute: %s", cudaGetErrorString(x)); return fail(YF_ERR_CUDA); }
    int rc = alloc_post(ctx);
    if (rc != YF_OK) return fail(rc);
    *out = ctx;
    return YF_OK;
}

extern "C" void yf_destroy(yf_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (float* p : ctx->d_act) cudaFree(p);
    cudaFree(ctx->d_w); cudaFree(ctx->d_skip); cudaFree(ctx->d_hl); cudaFree(ctx->d_hs); cudaFree(ctx->d_x); cudaFree(ctx->d_u8);
    cudaFree(ctx->d_out); cudaFree(ctx->d_counts); cudaFree(ctx->d_status);
    cudaFree(ctx->p_rec); cudaFree(ctx->p_conf); cudaFree(ctx->p_cls); cudaFree(ctx->p_sbox); cudaFree(ctx->p_order);
    cudaFree(ctx->p_alive); cudaFree(ctx->n_alive); cudaFree(ctx->prep_tab); cudaFree(ctx->d_bgr);
    cudaFree(ctx->d_coef); cudaFree(ctx->d_jframes); cudaFree(ctx->d_jstatus);
    cudaFree(ctx->d_jenc); cudaFree(ctx->d_jhdr); cudaFree(ctx->d_jout); cudaFree(ctx->d_jpack); cudaFree(ctx->d_jlen);
    for (auto& kv : ctx->graphs) cudaGraphExecDestroy(kv.second.first);
    if (ctx->s_cap) cudaStreamDestroy(ctx->s_cap);
    if (ctx->s_side) cudaStreamDestroy(ctx->s_side);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->s_copy) {
        cudaStreamSynchronize(ctx->s_copy); cudaStreamSynchronize(ctx->s_comp); cudaStreamSynchronize(ctx->s_back);
        for (int i = 0; i < 2; ++i) {
            cudaFree(ctx->sl_u8[i]); cudaFree(ctx->sl_out[i]); cudaFree(ctx->sl_counts[i]); cudaFree(ctx->sl_status[i]);
            cudaEventDestroy(ctx->sl_in[i]); cudaEventDestroy(ctx->sl_free[i]); cudaEventDestroy(ctx->sl_done[i]);
        }
        cudaStreamDestroy(ctx->s_copy); cudaStreamDestroy(ctx->s_comp); cudaStreamDestroy(ctx->s_back);
    }
    delete ctx;
}

extern "C" int yf_load_weights(yf_ctx* ctx, const float* host_blob, int64_t n_floats) {
    CTX_CHECK(ctx);
    if (!host_blob || n_floats != ctx->specs.total) {
        set_err(&ctx->err, "weight blob has %lld floats, expected %lld", (long long)n_floats, (long long)ctx->specs.total);
        return YF_ERR_ARG;
    }
    for (int64_t i = 0; i < n_floats; ++i)
        if (!std::isfinite(host_blob[i])) { set_err(&ctx->err, "non-finite weight at %lld", (long long)i); return YF_ERR_ARG; }
    CU(cudaSetDevice(ctx->device));
    if (ctx->groups.empty()) {                      // first weights: the forward's buffers and launch plan come into being now
        int rc = alloc_forward(ctx);
        if (rc != YF_OK) return rc;
        build_plan(ctx);
        set_sm_count(ctx);
    }
    Folded f{host_blob, &ctx->specs};
    std::vector<float>& P = ctx->host_packed;
    P.clear();
    std::vector<int64_t> offs;
    std::map<size_t, int64_t> offs2;                 // group index -> offset of its second weight block
    auto res = [&](auto tag, const std::string& n) {
        using C = decltype(tag);
        offs.push_back(pack_irb<C>(P, f, n + ".conv1", n + ".conv2", n + ".conv3", "", 0));
    };
    offs.push_back(ctx->in_ch == 3 ? pack_stem<CfgStem3>(P, f) : YF_USE_WIRB ? pack_wstem<CfgStemW>(P, f) : pack_stem<CfgStem>(P, f));
#if YF_USE_WIRB
    offs.push_back(pack_wirb<CfgRes1W>(P, f, "res1_1.conv1", "res1_1.conv2", "res1_1.conv3"));
#else
    res(CfgRes1{}, "res1_1");
#endif
    offs.push_back(YF_DENSE_TC ? pack_dense_tc(P, f) : pack_dense(P, f));
    {
        DenseSmall& d = ctx->dense_small;
        for (int c = 0; c < 24; ++c) {
            for (int k = 0; k < 4; ++k) d.w8[k][c] = f.w("conv1_8")[c * 4 + k];
            d.b8[c] = f.b("conv1_8")[c]; d.b9[c] = f.b("conv1_9")[c];
            for (int j = 0; j < 8; ++j) d.w21[c][j] = f.w("conv2_1")[j * 24 + c];
        }
        for (int j = 0; j < 8; ++j) d.b21[j] = f.b("conv2_1")[j];
    }
#if YF_USE_WIRB
    offs.push_back(pack_wirb<CfgRes2W>(P, f, "res2_1.conv1", "res2_1.conv2", "res2_1.conv3"));
    offs.push_back(pack_wirb<CfgRes2W>(P, f, "res2_2.conv1", "res2_2.conv2", "res2_2.conv3"));
    offs.push_back(pack_wirb<CfgDown2W>(P, f, "conv2_2", "conv2_3", "conv3_1"));
#else
    res(CfgRes2{}, "res2_1"); res(CfgRes2{}, "res2_2");
    offs.push_back(pack_irb<CfgDown2>(P, f, "conv2_2", "conv2_3", "conv3_1", "", 0));
#endif
    if (YF_USE_TC && YF_USE_TCT_A) {
        offs.push_back(pack_irbt<CfgRes3aTt>(P, f, "res3_1.conv1", "res3_1.conv2", "res3_1.conv3"));
        offs.push_back(pack_irbt<CfgRes3aTt>(P, f, "res3_2.conv1", "res3_2.conv2", "res3_2.conv3"));
    } else { res(CfgRes3a{}, "res3_1"); res(CfgRes3a{}, "res3_2"); }
    offs.push_back(ctx->variant == YF_VARIANT_LITE ? pack_lite34(P, f)
                   : (YF_USE_TC && YF_USE_TCT_A) ? pack_irbt<CfgWide3Tt>(P, f, "conv3_2", "conv3_3", "conv3_4")
                                                 : pack_irb<CfgWide3>(P, f, "conv3_2", "conv3_3", "conv3_4", "", 0));
#if YF_USE_TC
    for (const char* n : {"res3_3", "res3_4", "res3_5", "res3_6"})
        offs.push_back(YF_USE_TCT ? pack_irbt<CfgRes3bTt>(P, f, std::string(n) + ".conv1", std::string(n) + ".conv2", std::string(n) + ".conv3")
                                  : pack_irbtc<CfgRes3bTc>(P, f, std::string(n) + ".conv1", std::string(n) + ".conv2", std::string(n) + ".conv3"));
#else
    res(CfgRes3b{}, "res3_3"); res(CfgRes3b{}, "res3_4"); res(CfgRes3b{}, "res3_5"); res(CfgRes3b{}, "res3_6");
#endif
    offs.push_back((YF_USE_TC && YF_USE_TCT_A) ? pack_irbt<CfgDown3Tt>(P, f, "conv3_5", "conv3_6", "conv4_1") : pack_irb<CfgDown3>(P, f, "conv3_5", "conv3_6", "conv4_1", "", 0));
#if YF_USE_TC
    for (const char* n : {"res4_1", "res4_2", "res4_3", "res4_4"})
    {
        offs.push_back(pack_irbtc<CfgRes4Tc>(P, f, std::string(n) + ".conv1", std::string(n) + ".conv2", std::string(n) + ".conv3"));
        if (YF_USE_TCT) offs2[offs.size() - 1] = pack_irbt<CfgRes4Tt>(P, f, std::string(n) + ".conv1", std::string(n) + ".conv2", std::string(n) + ".conv3");
    }
#else
    res(CfgRes4{}, "res4_1"); res(CfgRes4{}, "res4_2"); res(CfgRes4{}, "res4_3"); res(CfgRes4{}, "res4_4");
#endif
    offs.push_back(pack_irb<CfgDown4>(P, f, "conv4_2", "conv4_3", "conv5_1", "", 0));
    if (YF_USE_TC && YF_USE_TCT_A) offs2[offs.size() - 1] = pack_irbt<CfgDown4Tt>(P, f, "conv4_2", "conv4_3", "conv5_1");
#if YF_RES5_TC
    for (const char* n : {"res5_1", "res5_2", "res5_3", "res5_4", "res5_5"})
        offs.push_back(pack_irbtc2<CfgRes5Tc>(P, f, std::string(n) + ".conv1", std::string(n) + ".conv2", std::string(n) + ".conv3"));
#else
    res(CfgRes5{}, "res5_1"); res(CfgRes5{}, "res5_2"); res(CfgRes5{}, "res5_3"); res(CfgRes5{}, "res5_4"); res(CfgRes5{}, "res5_5");
#endif
    offs.push_back(pack_pw52(P, f));
#if YF_USE_TC
    offs.push_back(pack_dwpwtc<CfgNeckS1Tc>(P, f, "conv5_3", "conv5_4"));
#else
    offs.push_back(pack_irb<CfgNeckS1>(P, f, "", "conv5_3", "conv5_4", "", 0));
#endif
    offs.push_back(heads_on_tc(ctx->nout) ? pack_dwpwtc_head<CfgNeckS2Tc>(P, f, "conv5_5", "conv5_6", "head_5", 128, ctx->nout)
                                          : pack_irb<CfgNeckS2>(P, f, "", "conv5_5", "conv5_6", "head_5", ctx->nout));
    if (ctx->variant != YF_VARIANT_LITE) {
    offs.push_back(upcat_on_tc(ctx->H, ctx->W) ? pack_upcat_tc(P, f) : pack_upcat(P, f));
#if YF_USE_TC
    offs.push_back(pack_dwpwtc<CfgNeckL1Tc>(P, f, "conv4_1_2", "conv4_1_3"));
#else
    offs.push_back(pack_irb<CfgNeckL1>(P, f, "", "conv4_1_2", "conv4_1_3", "", 0));
#endif
    offs.push_back(heads_on_tc(ctx->nout) ? pack_dwpwtc_head<CfgNeckL2Tc>(P, f, "conv4_1_4", "conv4_1_5", "head_4", 96, ctx->nout)
                                          : pack_irb<CfgNeckL2>(P, f, "", "conv4_1_4", "conv4_1_5", "head_4", ctx->nout));
    }
    pad4(P);
    if (offs.size() != ctx->groups.size()) { set_err(&ctx->err, "internal: %zu packs vs %zu groups", offs.size(), ctx->groups.size()); return YF_ERR_STATE; }
    for (auto& kv : ctx->graphs) cudaGraphExecDestroy(kv.second.first);      // graphs bake the weight pointers in
    ctx->graphs.clear();
    if (ctx->d_w) CU(cudaFree(ctx->d_w));
    ctx->d_w = nullptr;
    CU(cudaMalloc(&ctx->d_w, sizeof(float) * P.size()));
    CU(cudaMemcpy(ctx->d_w, P.data(), sizeof(float) * P.size(), cudaMemcpyHostToDevice));
    for (size_t i = 0; i < offs.size(); ++i) { ctx->groups[i].w_off = offs[i]; ctx->groups[i].a.w = ctx->d_w + offs[i]; }
    for (const auto& kv : offs2) ctx->groups[kv.first].a.w2 = ctx->d_w + kv.second;
    ctx->weights_loaded = true;
    return YF_OK;
}

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch pays where the launches are latency chains: measured (tools/pdl_ab.sh, profiles/r02_pdl_ab.txt) 0.369 -> 0.329 ms
// per batch-1 yf_detect on a stream, nothing inside a replayed CUDA graph (no launch gaps to hide), and -1.3% at batch 256 (the next
// kernel's CTAs take the slots of the finishing ones early and then only wait). So: small batches only. YF_PDL_MAX overrides (0 = never).
static bool pdl_enabled(int B) {
    static const int pdl_max = getenv("YF_PDL_MAX") ? atoi(getenv("YF_PDL_MAX")) : 16;
    return B <= pdl_max;
}
static const int kForkMaxBatch = 128;   // measured: -9% at batch 1, -2% at 64, -1% at 128, neutral at 256
static int forward_impl(yf_ctx* ctx, const void* x, bool u8in, int B, float* head_large, float* head_small, cudaStream_t st) {
    if (!ctx->weights_loaded) { set_err(&ctx->err, "yf_load_weights has not been called"); return YF_ERR_STATE; }
    if (B < 1 || B > ctx->max_batch) { set_err(&ctx->err, "batch %d outside [1, max_batch=%d]", B, ctx->max_batch); return YF_ERR_STATE; }
    if (!x || !head_small || (!head_large && ctx->variant != YF_VARIANT_LITE)) { set_err(&ctx->err, "null tensor pointer"); return YF_ERR_ARG; }
    static const bool debug_sync = getenv("YF_DEBUG_SYNC") != nullptr;
    // Small batches leave most SMs idle in the low-resolution groups, so the two head branches (yolo_fastest.py:203-216: conv5_3..head_5
    // and deconv5_1..head_4, both fed by conv5_2) run side by side: fork after conv5_2, join before the caller's next work. Large
    // batches fill the GPU with every kernel and stay on one stream.
    static const bool no_fork = getenv("YF_NO_FORK") != nullptr;
    static const int fork_max = getenv("YF_FORK_MAX") ? atoi(getenv("YF_FORK_MAX")) : kForkMaxBatch;
    const bool fork = B <= fork_max && !no_fork;
    if (fork && !ctx->s_side) {
        CU(cudaStreamCreateWithFlags(&ctx->s_side, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    }
    for (Group& g : ctx->groups) {
        GroupArgs a = g.a;
        const bool h5 = !strcmp(g.name, "head_5"), side = fork && (h5 || !strcmp(g.name, "conv5_4"));
        if (h5) a.y = head_small;
        if (!strcmp(g.name, "head_4")) a.y = head_large;
        if (side && !h5) {
            CU(cudaEventRecord(ctx->ev_fork, st));
            CU(cudaStreamWaitEvent(ctx->s_side, ctx->ev_fork, 0));
        }
        a.pdl = pdl_enabled(B) && !(side && !h5);          // not behind an event wait (the first launch of the side stream)
        g.launch(a, x, u8in, B, side ? ctx->s_side : st);
        if (side && h5) CU(cudaEventRecord(ctx->ev_join, ctx->s_side));
        ctx->launches++;
        if (debug_sync) {   // YF_DEBUG_SYNC=1: attribute a device fault to the group that raised it
            cudaError_t e = cudaStreamSynchronize(st);
            if (e == cudaSuccess) e = cudaGetLastError();
            if (e != cudaSuccess) {
                set_err(&ctx->err, "group '%s' failed: %s", g.name, cudaGetErrorString(e));
                return YF_ERR_CUDA;
            }
        }
    }
    if (fork) CU(cudaStreamWaitEvent(st, ctx->ev_join, 0));
    ctx->last_forward_forked = fork;
    CU(cudaGetLastError());
    for (Group& g : ctx->groups)
        if (g.tcache.failed) { set_err(&ctx->err, "cuTensorMapEncodeTiled failed for group '%s'", g.name); g.tcache.ptr = nullptr; return YF_ERR_CUDA; }
    return YF_OK;
}

// The asynchronous slot path (yf_detect_submit_u8*) runs on internal streams and shares the activations and the post-processing
// workspace with the blocking entry points, which run on the caller's stream: every blocking entry point first makes its stream wait
// for the slots in flight (a device-side dependency, no host block), so the two never overlap on those buffers.
static int order_after_slots(yf_ctx* ctx, cudaStream_t st) {
    for (int i = 0; i < 2; ++i)
        if (ctx->sl_used[i]) CU(cudaStreamWaitEvent(st, ctx->sl_done[i], 0));
    return YF_OK;
}
#define ORDER(ctx, st) do { int rc__ = order_after_slots(ctx, (cudaStream_t)(st)); if (rc__) return rc__; } while (0)

extern "C" int yf_forward(yf_ctx* ctx, const float* x, int B, float* head_large, float* head_small, void* stream) {
    CTX_CHECK(ctx);
    ORDER(ctx, stream);
    return forward_impl(ctx, x, false, B, head_large, head_small, (cudaStream_t)stream);
}

extern "C" int yf_tap(yf_ctx* ctx, const char* name, int B, float* dst, int64_t* per_image, void* stream) {
    CTX_CHECK(ctx);
    auto it = ctx->taps.find(name ? name : "");
    if (it == ctx->taps.end()) { set_err(&ctx->err, "no tap named '%s'", name ? name : "(null)"); return YF_ERR_ARG; }
    if (per_image) *per_image = it->second.second;
    if (dst) {
        if (B < 1 || B > ctx->max_batch) { set_err(&ctx->err, "bad batch %d", B); return YF_ERR_STATE; }
        CU(cudaMemcpyAsync(dst, it->second.first, sizeof(float) * it->second.second * B, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    }
    return YF_OK;
}

extern "C" int yf_profile_forward(yf_ctx* ctx, const float* x, int B, const char** names, float* ms, int cap) {
    CTX_CHECK(ctx);
    if (!ctx->weights_loaded) { set_err(&ctx->err, "weights not loaded"); return YF_ERR_STATE; }
    if (B < 1 || B > ctx->max_batch || !x) { set_err(&ctx->err, "bad arguments"); return YF_ERR_ARG; }
    ORDER(ctx, 0);
    const int n = (int)ctx->groups.size();
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto& e : ev) CU(cudaEventCreate(&e));
    for (int rep = 0; rep < 2; ++rep) {   // first pass warms up, second is reported
        CU(cudaEventRecord(ev[0], 0));
        for (int i = 0; i < n; ++i) {
            Group& g = ctx->groups[i];
            GroupArgs a = g.a;
            if (!strcmp(g.name, "head_5")) a.y = ctx->d_hs;
            if (!strcmp(g.name, "head_4")) a.y = ctx->d_hl;
            g.launch(a, x, false, B, 0);
            ctx->launches++;
            CU(cudaEventRecord(ev[i + 1], 0));
        }
        CU(cudaDeviceSynchronize());
    }
    int w = 0;
    for (int i = 0; i < n && w < cap; ++i, ++w) {
        float t = 0.f;
        CU(cudaEventElapsedTime(&t, ev[i], ev[i + 1]));
        if (names) names[w] = ctx->groups[i].name;
        if (ms) ms[w] = t;
    }
    for (auto& e : ev) cudaEventDestroy(e);
    return w;
}

#ifdef YF_TC_TRACE
// debug builds only: copy the phase trace of the last tensor-core launch (16 slots x 64 steps of clock64) to the host
extern "C" int yf_debug_trace(long long* dst, int n) {
    return (int)cudaMemcpyFromSymbol(dst, yf::g_tc_trace, sizeof(long long) * (size_t)(n < 16 * 64 ? n : 16 * 64));
}
#endif

// ---------------------------------------------------------------------------------------------
// post-processing
// ---------------------------------------------------------------------------------------------
// shared-memory sort capacity of the head kernel for NC candidates: the next power of two, 12 bytes per key; beyond 16 384 keys
// (196 KB) the kernel falls back to its global-memory rank
static int post_sort_cap(int NC) {
    int p2 = 32;
    while (p2 < NC) p2 <<= 1;
    return p2 <= 16384 ? p2 : 0;
}

static int post_impl(yf_ctx* ctx, const float* hl, const float* hs, int B, int hlh, int hlw, int hsh, int hsw,
                     const yf_post_params* p, yf_det* out, int32_t* counts, int32_t* status, int do_nms, cudaStream_t st) {
    if (!p || !hl || !hs || !out || !counts) { set_err(&ctx->err, "null argument"); return YF_ERR_ARG; }
    if (B < 1 || B > ctx->max_batch) { set_err(&ctx->err, "batch %d outside [1, max_batch=%d]", B, ctx->max_batch); return YF_ERR_STATE; }
    if (p->mode != YF_MODE_DETECT && p->mode != YF_MODE_VALIDATE) { set_err(&ctx->err, "bad mode %d", p->mode); return YF_ERR_ARG; }
    if (p->max_det < 1) { set_err(&ctx->err, "max_det must be >= 1"); return YF_ERR_ARG; }
    const int NC = ctx->num_anchors * (hlh * hlw + hsh * hsw);
    if (NC > ctx->NC || NC < 1) { set_err(&ctx->err, "%d candidates exceed the ctx capacity %d (created for %dx%d)", NC, ctx->NC, ctx->H, ctx->W); return YF_ERR_STATE; }
    PostArgs a;
    memset(&a, 0, sizeof a);
    a.head[0] = hl; a.head[1] = hs;
    a.A = ctx->num_anchors; a.nc = ctx->num_cls;
    a.h[0] = hlh; a.w[0] = hlw; a.h[1] = hsh; a.w[1] = hsw;
    memcpy(a.anchors, p->anchors, sizeof a.anchors);
    a.conf_thres = p->conf_thres; a.nms_thres = p->nms_thres;
    a.input_h = p->input_h; a.input_w = p->input_w; a.mode = p->mode; a.max_det = p->max_det; a.do_nms = do_nms;
    a.out = out; a.counts = counts; a.status = status;
    a.NC = NC;
    a.rec = ctx->p_rec; a.conf = ctx->p_conf; a.cls = ctx->p_cls; a.sbox = ctx->p_sbox; a.order = ctx->p_order; a.alive = ctx->p_alive;
    a.sort_cap = post_sort_cap(NC);
    // programmatic launch behind the last forward kernel of this stream, unless the forward forked (the join is an event dependency)
    const bool pdl = pdl_enabled(B) && !ctx->last_forward_forked;
    if (p->mode == YF_MODE_DETECT) launch_k(pdl, post_kernel<YF_MODE_DETECT>, B, POST_NT, (size_t)a.sort_cap * 12, st, a);
    else launch_k(pdl, post_kernel<YF_MODE_VALIDATE>, B, POST_NT, (size_t)a.sort_cap * 12, st, a);
    ctx->launches++;
    CU(cudaGetLastError());
    return YF_OK;
}

extern "C" int yf_postprocess(yf_ctx* ctx, const float* head_large, const float* head_small, int B, int hl, int wl, int hs, int ws,
                              const yf_post_params* p, yf_det* out, int32_t* counts, int32_t* status, void* stream) {
    CTX_CHECK(ctx);
    ORDER(ctx, stream);
    return post_impl(ctx, head_large, head_small, B, hl, wl, hs, ws, p, out, counts, status, 1, (cudaStream_t)stream);
}

extern "C" int yf_decode(yf_ctx* ctx, const float* head_large, const float* head_small, int B, int hl, int wl, int hs, int ws,
                         const yf_post_params* p, yf_det* out, int32_t* counts, int32_t* status, void* stream) {
    CTX_CHECK(ctx);
    ORDER(ctx, stream);
    return post_impl(ctx, head_large, head_small, B, hl, wl, hs, ws, p, out, counts, status, 0, (cudaStream_t)stream);
}

extern "C" int yf_val_decode(yf_ctx* ctx, const float* head, int B, int h, int w, const double* anchors, int num_anchors,
                             int num_cls, int input_h, int input_w, float* out, void* stream) {
    CTX_CHECK(ctx);
    if (!head || !anchors || !out || B < 1 || h < 1 || w < 1 || num_anchors < 1 || num_anchors > YF_MAX_ANCHORS || num_cls < 1) {
        set_err(&ctx->err, "bad argument"); return YF_ERR_ARG;
    }
    ValDecodeArgs a;
    a.head = head; a.out = out; a.B = B; a.A = num_anchors; a.nc = num_cls; a.h = h; a.w = w;
    const double sw = (double)input_w / (double)w, sh = (double)input_h / (double)h;
    a.stride_w = (float)sw; a.stride_h = (float)sh;
    for (int i = 0; i < num_anchors; ++i) { a.aw[i] = (float)(anchors[2 * i] / sw); a.ah[i] = (float)(anchors[2 * i + 1] / sh); }
    const long long total = (long long)B * num_anchors * h * w;
    val_decode_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
    ctx->launches++;
    CU(cudaGetLastError());
    return YF_OK;
}

extern "C" int yf_val_nms(yf_ctx* ctx, const float* pred, int B, int N, double conf_thres, double nms_thres, int max_det,
                          yf_det* out, int32_t* counts, int32_t* status, void* stream) {
    CTX_CHECK(ctx);
    if (!pred || !out || !counts || max_det < 1) { set_err(&ctx->err, "bad argument"); return YF_ERR_ARG; }
    if (B < 1 || B > ctx->max_batch) { set_err(&ctx->err, "batch %d outside [1, max_batch=%d]", B, ctx->max_batch); return YF_ERR_STATE; }
    if (N < 1 || N > ctx->NC) { set_err(&ctx->err, "%d rows exceed the ctx capacity %d", N, ctx->NC); return YF_ERR_STATE; }
    ORDER(ctx, stream);
    PostArgs a;
    memset(&a, 0, sizeof a);
    a.pred = pred;
    a.A = ctx->num_anchors; a.nc = ctx->num_cls;
    a.conf_thres = conf_thres; a.nms_thres = nms_thres;
    a.mode = YF_MODE_VALIDATE; a.max_det = max_det; a.do_nms = 1;
    a.out = out; a.counts = counts; a.status = status;
    a.NC = N;
    a.rec = ctx->p_rec; a.conf = ctx->p_conf; a.cls = ctx->p_cls; a.sbox = ctx->p_sbox; a.order = ctx->p_order; a.alive = ctx->p_alive;
    a.sort_cap = post_sort_cap(N);
    post_kernel<POST_SRC_ROWS><<<B, POST_NT, a.sort_cap * 12, (cudaStream_t)stream>>>(a);
    ctx->launches++;
    CU(cudaGetLastError());
    return YF_OK;
}

static int nms_scratch(yf_ctx* ctx, int n) {
    if (n <= ctx->n_alive_cap) return YF_OK;
    if (ctx->n_alive) CU(cudaFree(ctx->n_alive));
    ctx->n_alive = nullptr;
    CU(cudaMalloc(&ctx->n_alive, (size_t)n));
    ctx->n_alive_cap = n;
    return YF_OK;
}

extern "C" int yf_nms_sorted_i32(yf_ctx* ctx, const int32_t* boxes, int n, double nms_thres, int32_t* keep, int32_t* n_keep, void* stream) {
    CTX_CHECK(ctx);
    if (!boxes || !keep || !n_keep || n < 0) { set_err(&ctx->err, "bad argument"); return YF_ERR_ARG; }
    int rc = nms_scratch(ctx, n > 0 ? n : 1);
    if (rc) return rc;
    nms_sorted_kernel<YF_MODE_DETECT><<<1, 32, 0, (cudaStream_t)stream>>>(reinterpret_cast<const int4*>(boxes), ctx->n_alive, n, nms_thres, 0.f, keep, n_keep);
    ctx->launches++;
    CU(cudaGetLastError());
    return YF_OK;
}

extern "C" int yf_nms_sorted_f32(yf_ctx* ctx, const float* boxes_f, int n, float nms_thres, int32_t* keep, int32_t* n_keep, void* stream) {
    CTX_CHECK(ctx);
    if (!boxes_f || !keep || !n_keep || n < 0) { set_err(&ctx->err, "bad argument"); return YF_ERR_ARG; }
    int rc = nms_scratch(ctx, n > 0 ? n : 1);
    if (rc) return rc;
    nms_sorted_kernel<YF_MODE_VALIDATE><<<1, 32, 0, (cudaStream_t)stream>>>(reinterpret_cast<const int4*>(boxes_f), ctx->n_alive, n, 0.0, nms_thres, keep, n_keep);
    ctx->launches++;
    CU(cudaGetLastError());
    return YF_OK;
}

// ---------------------------------------------------------------------------------------------
// fused paths
// ---------------------------------------------------------------------------------------------
static int detect_impl(yf_ctx* ctx, const void* x, bool u8in, int B, const yf_post_params* p, yf_det* out, int32_t* counts,
                       int32_t* status, cudaStream_t st) {
    int rc = forward_impl(ctx, x, u8in, B, ctx->d_hl, ctx->d_hs, st);
    if (rc) return rc;
    return post_impl(ctx, ctx->d_hl, ctx->d_hs, B, ctx->H / 16, ctx->W / 16, ctx->H / 32, ctx->W / 32, p, out, counts, status, 1, st);
}

extern "C" int yf_detect(yf_ctx* ctx, const float* x, int B, const yf_post_params* p, yf_det* out, int32_t* counts,
                         int32_t* status, void* stream) {
    CTX_CHECK(ctx);
    ORDER(ctx, stream);
    return detect_impl(ctx, x, false, B, p, out, counts, status, (cudaStream_t)stream);
}

// detect_impl on library-owned buffers, replayed from a CUDA graph for small batches (31 launches cost more on the
// host than on the device at batch 1). The graph is keyed by everything baked into the kernel arguments.
static const int kGraphMaxBatch = 16;
static int detect_fixed(yf_ctx* ctx, const void* xdev, bool u8in, int B, const yf_post_params* p, yf_det* out, int32_t* counts,
                        int32_t* status, cudaStream_t st) {
    static const bool no_graph = getenv("YF_DEBUG_SYNC") != nullptr || getenv("YF_NO_GRAPH") != nullptr;
    if (B > kGraphMaxBatch || no_graph) return detect_impl(ctx, xdev, u8in, B, p, out, counts, status, st);
    std::string key(reinterpret_cast<const char*>(p), sizeof(*p));
    const void* ptrs[4] = {xdev, out, counts, status};
    key.append(reinterpret_cast<const char*>(ptrs), sizeof ptrs);
    key.push_back((char)B); key.push_back((char)u8in);
    auto it = ctx->graphs.find(key);
    if (it == ctx->graphs.end()) {
        if (!ctx->weights_loaded) { set_err(&ctx->err, "yf_load_weights has not been called"); return YF_ERR_STATE; }
        cudaGraph_t graph = nullptr;
        cudaGraphExec_t exec = nullptr;
        const int64_t before = ctx->launches;
        if (!ctx->s_cap) CU(cudaStreamCreateWithFlags(&ctx->s_cap, cudaStreamNonBlocking));
        CU(cudaStreamBeginCapture(ctx->s_cap, cudaStreamCaptureModeThreadLocal));
        int rc = detect_impl(ctx, xdev, u8in, B, p, out, counts, status, ctx->s_cap);
        cudaError_t e = cudaStreamEndCapture(ctx->s_cap, &graph);
        const int n = (int)(ctx->launches - before);
        ctx->launches = before;                              // captured, not executed
        if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (e != cudaSuccess) { set_err(&ctx->err, "graph capture failed: %s", cudaGetErrorString(e)); return YF_ERR_CUDA; }
        CU(cudaGraphInstantiate(&exec, graph, 0));
        cudaGraphDestroy(graph);
        it = ctx->graphs.emplace(key, std::make_pair(exec, n)).first;
    }
    CU(cudaGraphLaunch(it->second.first, st));
    ctx->launches += it->second.second;
    return YF_OK;
}

static int detect_host_impl(yf_ctx* ctx, const void* x_host, bool u8in, int B, const yf_post_params* p, yf_det* out_host,
                            int32_t* counts_host, int32_t* status_host, cudaStream_t st) {
    if (!x_host || !p || !out_host || !counts_host) { set_err(&ctx->err, "null argument"); return YF_ERR_ARG; }
    if (B < 1 || B > ctx->max_batch) { set_err(&ctx->err, "batch %d outside [1, max_batch=%d]", B, ctx->max_batch); return YF_ERR_STATE; }
    if (p->max_det < 1) { set_err(&ctx->err, "max_det must be >= 1"); return YF_ERR_ARG; }
    CU(cudaSetDevice(ctx->device));
    if (!ctx->weights_loaded) { set_err(&ctx->err, "yf_load_weights has not been called"); return YF_ERR_STATE; }
    ORDER(ctx, st);
    int rc = ensure_out(ctx, p->max_det);
    if (rc) return rc;
    const size_t npx = (size_t)B * ctx->in_ch * ctx->H * ctx->W;
    const void* xdev;
    if (u8in) { CU(cudaMemcpyAsync(ctx->d_u8, x_host, npx, cudaMemcpyHostToDevice, st)); xdev = ctx->d_u8; }
    else { CU(cudaMemcpyAsync(ctx->d_x, x_host, npx * sizeof(float), cudaMemcpyHostToDevice, st)); xdev = ctx->d_x; }
    rc = detect_fixed(ctx, xdev, u8in, B, p, ctx->d_out, ctx->d_counts, ctx->d_status, st);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out_host, ctx->d_out, sizeof(yf_det) * (size_t)B * p->max_det, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(counts_host, ctx->d_counts, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    if (status_host) CU(cudaMemcpyAsync(status_host, ctx->d_status, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return YF_OK;
}

extern "C" int yf_detect_host(yf_ctx* ctx, const float* x_host, int B, const yf_post_params* p, yf_det* out_host,
                              int32_t* counts_host, int32_t* status_host, void* stream) {
    CTX_CHECK(ctx);
    return detect_host_impl(ctx, x_host, false, B, p, out_host, counts_host, status_host, (cudaStream_t)stream);
}

extern "C" int yf_detect_host_u8(yf_ctx* ctx, const uint8_t* u8_host, int B, const yf_post_params* p, yf_det* out_host,
                                 int32_t* counts_host, int32_t* status_host, void* stream) {
    CTX_CHECK(ctx);
    return detect_host_impl(ctx, u8_host, true, B, p, out_host, counts_host, status_host, (cudaStream_t)stream);
}

// ---- GPU pre-processing: BGR frames -> gray -> bilinear resize to the network input (detect.py:107-122) ------------------------
static int prep_enqueue(yf_ctx* ctx, const uint8_t* bgr_dev, int B, int Ho, int Wo, uint8_t* gray_dev, cudaStream_t st) {
    if (ctx->in_ch != 1) { set_err(&ctx->err, "pre-processing serves the single-channel models"); return YF_ERR_STATE; }
    if (Ho < 1 || Wo < 1 || Ho > 16384 || Wo > 16384) { set_err(&ctx->err, "source size %dx%d not supported", Ho, Wo); return YF_ERR_ARG; }
    if (Ho != ctx->prep_Ho || Wo != ctx->prep_Wo) {
        std::vector<PrepTap> tab((size_t)ctx->W + ctx->H);
        prep_taps(ctx->W, Wo, false, tab.data());
        prep_taps(ctx->H, Ho, true, tab.data() + ctx->W);
        if (!ctx->prep_tab) CU(cudaMalloc(&ctx->prep_tab, sizeof(PrepTap) * tab.size()));
        CU(cudaStreamSynchronize(st));                  // a kernel enqueued earlier may still read the old tables
        CU(cudaMemcpy(ctx->prep_tab, tab.data(), sizeof(PrepTap) * tab.size(), cudaMemcpyHostToDevice));
        ctx->prep_Ho = Ho; ctx->prep_Wo = Wo;
    }
    const int nsm = ctx->groups.empty() ? 148 : ctx->groups[0].a.nsm;
    const int W4 = ctx->W / 4, Wo4 = Wo / 4;
    const int nt = Wo4 > 0 && Wo4 <= 512 ? (512 / Wo4) * Wo4 : Wo4;       // staging threads: a whole number of frame rows
    const size_t smem = (size_t)2 * PREP_R * Wo;
    if (Wo % 4 == 0 && nt >= 32 && nt <= 1024 && W4 <= nt && smem <= 48 * 1024 && ((uintptr_t)bgr_dev & 3) == 0) {
        const long long groups = (long long)B * ((ctx->H + PREP_R - 1) / PREP_R);
        const int grid = (int)std::min<long long>(groups, (long long)nsm * (2048 / nt));
        prep_bgr_rows_kernel<<<grid, nt, smem, st>>>(bgr_dev, gray_dev, ctx->prep_tab, ctx->prep_tab + ctx->W, B, Ho, Wo, ctx->H, ctx->W);
    } else {                                            // any width / alignment: one thread per 4 output pixels, byte loads
        const long long total = (long long)B * ctx->H * W4;
        const int grid = (int)std::min<long long>((total + 255) / 256, (long long)nsm * 16);
        prep_bgr_kernel<<<grid, 256, 0, st>>>(bgr_dev, gray_dev, ctx->prep_tab, ctx->prep_tab + ctx->W, B, Ho, Wo, ctx->H, ctx->W);
    }
    CU(cudaGetLastError());
    ctx->launches += 1;
    return YF_OK;
}

// grow-only device staging of host frames (yf_detect_host_bgr / yf_detect_host_frames)
static int ensure_bgr(yf_ctx* ctx, size_t nbytes, cudaStream_t st) {
    if (nbytes <= ctx->bgr_cap) return YF_OK;
    CU(cudaStreamSynchronize(st));                      // an earlier call's kernels may still read the old buffer
    if (ctx->d_bgr) CU(cudaFree(ctx->d_bgr));
    ctx->d_bgr = nullptr; ctx->bgr_cap = 0;
    CU(cudaMalloc(&ctx->d_bgr, nbytes));
    ctx->bgr_cap = nbytes;
    return YF_OK;
}

extern "C" int yf_preprocess_bgr(yf_ctx* ctx, const uint8_t* bgr_dev, int B, int Ho, int Wo, uint8_t* gray_dev, void* stream) {
    CTX_CHECK(ctx);
    if (!bgr_dev || !gray_dev || B < 1) { set_err(&ctx->err, "bad argument"); return YF_ERR_ARG; }
    CU(cudaSetDevice(ctx->device));
    return prep_enqueue(ctx, bgr_dev, B, Ho, Wo, gray_dev, (cudaStream_t)stream);
}

extern "C" int yf_detect_host_bgr(yf_ctx* ctx, const uint8_t* bgr_host, int B, int Ho, int Wo, const yf_post_params* p,
                                  yf_det* out_host, int32_t* counts_host, int32_t* status_host, void* stream) {
    CTX_CHECK(ctx);
    cudaStream_t st = (cudaStream_t)stream;
    if (!bgr_host || !p || !out_host || !counts_host) { set_err(&ctx->err, "null argument"); return YF_ERR_ARG; }
    if (B < 1 || B > ctx->max_batch) { set_err(&ctx->err, "batch %d outside [1, max_batch=%d]", B, ctx->max_batch); return YF_ERR_STATE; }
    if (p->max_det < 1) { set_err(&ctx->err, "max_det must be >= 1"); return YF_ERR_ARG; }
    CU(cudaSetDevice(ctx->device));
    if (!ctx->weights_loaded) { set_err(&ctx->err, "yf_load_weights has not been called"); return YF_ERR_STATE; }
    ORDER(ctx, st);
    int rc = ensure_out(ctx, p->max_det);
    if (rc) return rc;
    const size_t nbytes = (size_t)B * Ho * Wo * 3;
    if ((rc = ensure_bgr(ctx, nbytes, st))) return rc;
    CU(cudaMemcpyAsync(ctx->d_bgr, bgr_host, nbytes, cudaMemcpyHostToDevice, st));
    rc = prep_enqueue(ctx, ctx->d_bgr, B, Ho, Wo, ctx->d_u8, st);
    if (rc) return rc;
    rc = detect_fixed(ctx, ctx->d_u8, true, B, p, ctx->d_out, ctx->d_counts, ctx->d_status, st);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out_host, ctx->d_out, sizeof(yf_det) * (size_t)B * p->max_det, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(counts_host, ctx->d_counts, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    if (status_host) CU(cudaMemcpyAsync(status_host, ctx->d_status, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return YF_OK;
}

// ---- frames of mixed sizes, gray or colour networks (one launch per PREP_CHUNK frames, taps computed in the kernel) --------------
static const int kPrepMaxSide = 16384;

// every descriptor against the size range and, when the buffer size is known (nbytes >= 0), against the buffer
static int frames_check(yf_ctx* ctx, int B, const int64_t* off, const int32_t* Ho, const int32_t* Wo, int64_t nbytes) {
    if (!off || !Ho || !Wo) { set_err(&ctx->err, "null descriptor array"); return YF_ERR_ARG; }
    if (B < 1 || B > ctx->max_batch) { set_err(&ctx->err, "batch %d outside [1, max_batch=%d]", B, ctx->max_batch); return YF_ERR_ARG; }
    for (int b = 0; b < B; ++b) {
        if (Ho[b] < 1 || Wo[b] < 1 || Ho[b] > kPrepMaxSide || Wo[b] > kPrepMaxSide) {
            set_err(&ctx->err, "frame %d: size %dx%d outside [1, %d]", b, Ho[b], Wo[b], kPrepMaxSide); return YF_ERR_ARG;
        }
        const int64_t size = (int64_t)Ho[b] * Wo[b] * 3;
        if (off[b] < 0 || (nbytes >= 0 && off[b] > nbytes - size)) {
            set_err(&ctx->err, "frame %d: bytes [%lld, %lld) outside the %lld-byte buffer", b, (long long)off[b], (long long)(off[b] + size),
                    (long long)nbytes);
            return YF_ERR_ARG;
        }
    }
    return YF_OK;
}

static int frames_enqueue(yf_ctx* ctx, const uint8_t* frames, int B, const int64_t* off, const int32_t* Ho, const int32_t* Wo,
                          uint8_t* out, cudaStream_t st) {
    const int nsm = ctx->groups.empty() ? 148 : ctx->groups[0].a.nsm;
    const long long groups = (ctx->H + PREP_R - 1) / PREP_R;
    const size_t per_img = (size_t)ctx->in_ch * ctx->H * ctx->W;
    PrepFrames fr;
    for (int c0 = 0; c0 < B; c0 += PREP_CHUNK) {
        const int n = std::min(PREP_CHUNK, B - c0);
        int smem = 0;                                   // from the widest frame of the chunk that is staged
        for (int i = 0; i < n; ++i) {
            fr.f[i] = {off[c0 + i], Ho[c0 + i], Wo[c0 + i]};
            if (prep_stageable(frames, fr.f[i], ctx->in_ch, PREP_SMEM_CAP)) smem = std::max(smem, prep_stage_bytes(fr.f[i].Wo, ctx->in_ch));
        }
        auto kern = ctx->in_ch == 1 ? prep_frames_kernel<1> : prep_frames_kernel<3>;
        int per_sm = 1;                                 // resident blocks: the grid strides over the rest
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, PREP_NT, smem));
        const int grid = (int)std::min<long long>((long long)n * groups, (long long)nsm * std::max(per_sm, 1));
        kern<<<grid, PREP_NT, smem, st>>>(frames, fr, n, out + c0 * per_img, ctx->H, ctx->W, smem);
        CU(cudaGetLastError());
        ctx->launches += 1;
    }
    return YF_OK;
}

extern "C" int yf_preprocess_frames(yf_ctx* ctx, const uint8_t* frames, int B, const int64_t* off, const int32_t* Ho, const int32_t* Wo,
                                    uint8_t* out, void* stream) {
    CTX_CHECK(ctx);
    if (!frames || !out) { set_err(&ctx->err, "null frames or output pointer"); return YF_ERR_ARG; }
    int rc = frames_check(ctx, B, off, Ho, Wo, -1);
    if (rc) return rc;
    CU(cudaSetDevice(ctx->device));
    return frames_enqueue(ctx, frames, B, off, Ho, Wo, out, (cudaStream_t)stream);
}

extern "C" int yf_detect_host_frames(yf_ctx* ctx, const uint8_t* frames_host, int64_t nbytes, int B, const int64_t* off, const int32_t* Ho,
                                     const int32_t* Wo, const yf_post_params* p, yf_det* out_host, int32_t* counts_host,
                                     int32_t* status_host, void* stream) {
    CTX_CHECK(ctx);
    cudaStream_t st = (cudaStream_t)stream;
    if (!frames_host || !p || !out_host || !counts_host) { set_err(&ctx->err, "null argument"); return YF_ERR_ARG; }
    if (p->max_det < 1) { set_err(&ctx->err, "max_det must be >= 1"); return YF_ERR_ARG; }
    int rc = frames_check(ctx, B, off, Ho, Wo, nbytes);
    if (rc) return rc;
    CU(cudaSetDevice(ctx->device));
    if (!ctx->weights_loaded) { set_err(&ctx->err, "yf_load_weights has not been called"); return YF_ERR_STATE; }
    ORDER(ctx, st);
    if ((rc = ensure_out(ctx, p->max_det))) return rc;
    if ((rc = ensure_bgr(ctx, (size_t)nbytes, st))) return rc;
    CU(cudaMemcpyAsync(ctx->d_bgr, frames_host, (size_t)nbytes, cudaMemcpyHostToDevice, st));      // the packed frames, one copy
    if ((rc = frames_enqueue(ctx, ctx->d_bgr, B, off, Ho, Wo, ctx->d_u8, st))) return rc;
    if ((rc = detect_fixed(ctx, ctx->d_u8, true, B, p, ctx->d_out, ctx->d_counts, ctx->d_status, st))) return rc;
    CU(cudaMemcpyAsync(out_host, ctx->d_out, sizeof(yf_det) * (size_t)B * p->max_det, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(counts_host, ctx->d_counts, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    if (status_host) CU(cudaMemcpyAsync(status_host, ctx->d_status, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return YF_OK;
}

// ---- baseline JPEG files decoded on the device (yf_jpeg.cuh): parse every header, one copy of the files, 3 launches per chunk ----------
extern "C" int yf_jpeg_probe(const uint8_t* data, int64_t nbytes, int32_t* h, int32_t* w) {
    JpegDesc d;
    std::string why;
    if (!jpeg_parse(data, nbytes, d, why)) { set_err(nullptr, "%s", why.c_str()); return YF_ERR_ARG; }
    if (h) *h = d.h;
    if (w) *w = d.w;
    return YF_OK;
}

// every file's bytes against the buffer, its header through the parser, and (frames_bytes >= 0) its frame against the output buffer
static int jpeg_check(yf_ctx* ctx, const uint8_t* files, int64_t nbytes, int B, const int64_t* off, const int64_t* len,
                      const int64_t* frame_off, int64_t frames_bytes, std::vector<JpegDesc>& ds) {
    if (!files || !off || !len || !frame_off) { set_err(&ctx->err, "null file or descriptor array"); return YF_ERR_ARG; }
    if (B < 1) { set_err(&ctx->err, "batch %d < 1", B); return YF_ERR_ARG; }
    ds.resize(B);
    std::string why;
    for (int b = 0; b < B; ++b) {
        if (off[b] < 0 || len[b] < 1 || off[b] > nbytes - len[b]) {
            set_err(&ctx->err, "file %d: bytes [%lld, %lld) outside the %lld-byte buffer", b, (long long)off[b], (long long)(off[b] + len[b]),
                    (long long)nbytes);
            return YF_ERR_ARG;
        }
        if (!jpeg_parse(files + off[b], len[b], ds[b], why)) { set_err(&ctx->err, "file %d: %s", b, why.c_str()); return YF_ERR_ARG; }
        const int64_t size = (int64_t)ds[b].h * ds[b].w * 3;
        if (frame_off[b] < 0 || (frames_bytes >= 0 && frame_off[b] > frames_bytes - size)) {
            set_err(&ctx->err, "frame %d: bytes [%lld, %lld) outside the %lld-byte frame buffer", b, (long long)frame_off[b],
                    (long long)(frame_off[b] + size), (long long)frames_bytes);
            return YF_ERR_ARG;
        }
        ds[b].src = off[b];
        ds[b].dst = frame_off[b];
    }
    return YF_OK;
}

// Files per warp of the entropy kernel: 1 (the default, DESIGN.md §5.7) or 32; YF_JPEG_FILES_PER_WARP selects the other for timing.
static int jpeg_fpw() {
    const char* e = getenv("YF_JPEG_FILES_PER_WARP");
    return e && atoi(e) == 32 ? 32 : 1;
}

// files dev (staged) -> frames dev, status dev [B]. The coefficient workspace holds one chunk and is reused in stream order.
static int jpeg_enqueue(yf_ctx* ctx, const uint8_t* files, std::vector<JpegDesc>& ds, uint8_t* frames, int32_t* status, cudaStream_t st) {
    const int B = (int)ds.size();
    int64_t most = 0;
    for (int c0 = 0; c0 < B; c0 += JPEG_CHUNK) {
        int64_t blocks = 0;
        for (int i = c0; i < std::min(B, c0 + JPEG_CHUNK); ++i) { ds[i].cbase = blocks; blocks += jpeg_blocks(ds[i]); }
        most = std::max(most, blocks);
    }
    const size_t need = (size_t)most * 128;
    if (need > ctx->coef_cap) {
        CU(cudaStreamSynchronize(st));                  // an earlier call's kernels may still use the old workspace
        if (ctx->d_coef) CU(cudaFree(ctx->d_coef));
        ctx->d_coef = nullptr; ctx->coef_cap = 0;
        CU(cudaMalloc(&ctx->d_coef, need));
        ctx->coef_cap = need;
    }
    const int fpw = jpeg_fpw();
    JpegChunk ch;
    for (int c0 = 0; c0 < B; c0 += JPEG_CHUNK) {
        const int n = std::min(JPEG_CHUNK, B - c0);
        int64_t max_blocks = 1, max_px = 1;
        for (int i = 0; i < n; ++i) {
            ch.d[i] = ds[c0 + i];
            max_blocks = std::max(max_blocks, jpeg_blocks(ch.d[i]));
            max_px = std::max(max_px, (int64_t)ch.d[i].h * ch.d[i].w);
        }
        if (fpw == 32) jpeg_entropy_kernel<32><<<(n + 31) / 32, 32, 32 * JPEG_TABS_BYTES, st>>>(files, ch, n, ctx->d_coef, status + c0);
        else jpeg_entropy_kernel<1><<<n, 32, JPEG_TABS_BYTES, st>>>(files, ch, n, ctx->d_coef, status + c0);
        CU(cudaGetLastError());
        const dim3 gi((unsigned)std::min<int64_t>((max_blocks + JPEG_IDCT_NT - 1) / JPEG_IDCT_NT, 2048), (unsigned)n);
        jpeg_idct_kernel<<<gi, JPEG_IDCT_NT, 0, st>>>(files, ch, ctx->d_coef);
        CU(cudaGetLastError());
        const dim3 gc((unsigned)std::min<int64_t>((max_px + JPEG_COLOR_NT - 1) / JPEG_COLOR_NT, 4096), (unsigned)n);
        jpeg_color_kernel<<<gc, JPEG_COLOR_NT, 0, st>>>(ch, ctx->d_coef, frames);
        CU(cudaGetLastError());
        ctx->launches += 3;
    }
    return YF_OK;
}

extern "C" int yf_decode_jpeg(yf_ctx* ctx, const uint8_t* files_host, int64_t nbytes, int B, const int64_t* off, const int64_t* len,
                              uint8_t* frames_dev, const int64_t* frame_off, int64_t frames_bytes, int32_t* status_dev, void* stream) {
    CTX_CHECK(ctx);
    cudaStream_t st = (cudaStream_t)stream;
    if (!frames_dev || !status_dev) { set_err(&ctx->err, "null frames or status pointer"); return YF_ERR_ARG; }
    std::vector<JpegDesc> ds;
    int rc = jpeg_check(ctx, files_host, nbytes, B, off, len, frame_off, frames_bytes, ds);
    if (rc) return rc;
    CU(cudaSetDevice(ctx->device));
    if ((rc = ensure_bgr(ctx, (size_t)nbytes, st))) return rc;
    CU(cudaMemcpyAsync(ctx->d_bgr, files_host, (size_t)nbytes, cudaMemcpyHostToDevice, st));       // the files, one copy
    return jpeg_enqueue(ctx, ctx->d_bgr, ds, frames_dev, status_dev, st);
}

extern "C" int yf_detect_host_jpeg(yf_ctx* ctx, const uint8_t* files_host, int64_t nbytes, int B, const int64_t* off, const int64_t* len,
                                   const int64_t* frame_off, const yf_post_params* p, yf_det* out_host, int32_t* counts_host,
                                   int32_t* status_host, uint8_t* frames_host, void* stream) {
    CTX_CHECK(ctx);
    cudaStream_t st = (cudaStream_t)stream;
    if (!p || !out_host || !counts_host) { set_err(&ctx->err, "null argument"); return YF_ERR_ARG; }
    if (p->max_det < 1) { set_err(&ctx->err, "max_det must be >= 1"); return YF_ERR_ARG; }
    if (B < 1 || B > ctx->max_batch) { set_err(&ctx->err, "batch %d outside [1, max_batch=%d]", B, ctx->max_batch); return YF_ERR_ARG; }
    std::vector<JpegDesc> ds;
    int rc = jpeg_check(ctx, files_host, nbytes, B, off, len, frame_off, -1, ds);
    if (rc) return rc;
    std::vector<int32_t> Ho(B), Wo(B);
    int64_t frames_bytes = 0;
    for (int b = 0; b < B; ++b) {
        Ho[b] = ds[b].h; Wo[b] = ds[b].w;
        frames_bytes = std::max(frames_bytes, frame_off[b] + (int64_t)Ho[b] * Wo[b] * 3);
    }
    CU(cudaSetDevice(ctx->device));
    if (!ctx->weights_loaded) { set_err(&ctx->err, "yf_load_weights has not been called"); return YF_ERR_STATE; }
    ORDER(ctx, st);
    if ((rc = ensure_out(ctx, p->max_det))) return rc;
    if ((rc = ensure_bgr(ctx, (size_t)nbytes, st))) return rc;
    if ((size_t)frames_bytes > ctx->jframes_cap) {
        CU(cudaStreamSynchronize(st));                  // an earlier call's kernels may still read the old frames
        if (ctx->d_jframes) CU(cudaFree(ctx->d_jframes));
        ctx->d_jframes = nullptr; ctx->jframes_cap = 0;
        CU(cudaMalloc(&ctx->d_jframes, (size_t)frames_bytes));
        ctx->jframes_cap = (size_t)frames_bytes;
    }
    if (!ctx->d_jstatus) CU(cudaMalloc(&ctx->d_jstatus, sizeof(int32_t) * ctx->max_batch));
    CU(cudaMemcpyAsync(ctx->d_bgr, files_host, (size_t)nbytes, cudaMemcpyHostToDevice, st));       // the files, one copy
    if ((rc = jpeg_enqueue(ctx, ctx->d_bgr, ds, ctx->d_jframes, ctx->d_jstatus, st))) return rc;
    if ((rc = frames_enqueue(ctx, ctx->d_jframes, B, frame_off, Ho.data(), Wo.data(), ctx->d_u8, st))) return rc;
    if ((rc = detect_fixed(ctx, ctx->d_u8, true, B, p, ctx->d_out, ctx->d_counts, ctx->d_status, st))) return rc;
    std::vector<int32_t> jst(B);
    CU(cudaMemcpyAsync(out_host, ctx->d_out, sizeof(yf_det) * (size_t)B * p->max_det, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(counts_host, ctx->d_counts, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    if (status_host) CU(cudaMemcpyAsync(status_host, ctx->d_status, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(jst.data(), ctx->d_jstatus, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    if (frames_host) CU(cudaMemcpyAsync(frames_host, ctx->d_jframes, (size_t)frames_bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int b = 0; b < B; ++b) {
        if (status_host) status_host[b] |= jst[b];
        else if (jst[b]) { set_err(&ctx->err, "file %d: corrupt entropy-coded data", b); return YF_ERR_DOMAIN; }
    }
    return YF_OK;
}

// ---- JPEG files encoded on the device (yf_jpeg_enc.cuh): headers built on the host, 4 launches per chunk of 256 frames ------------
static int jpeg_enc_params(std::string* err, int quality, int sampling, int& hs, int& vs) {
    if (quality < 1 || quality > 100) { set_err(err, "quality %d outside [1, 100]", quality); return YF_ERR_ARG; }
    if (!jpeg_enc_sampling(sampling, hs, vs)) {
        set_err(err, "sampling factor 0x%x is not supported (0x221111 4:2:0, 0x211111 4:2:2 and 0x111111 4:4:4 are)", sampling);
        return YF_ERR_ARG;
    }
    return YF_OK;
}

static bool jpeg_enc_size_ok(int h, int w) { return h >= 1 && w >= 1 && h <= JPEG_MAX_SIDE && w <= JPEG_MAX_SIDE; }

extern "C" int64_t yf_jpeg_encode_bound(int h, int w, int sampling) {
    int hs, vs;
    if (jpeg_enc_params(nullptr, 95, sampling, hs, vs)) return YF_ERR_ARG;
    if (!jpeg_enc_size_ok(h, w)) { set_err(nullptr, "size %dx%d outside [1, %d]", h, w, JPEG_MAX_SIDE); return YF_ERR_ARG; }
    return jpeg_enc_file_max(h, w, hs, vs);
}

extern "C" int yf_jpeg_encode_header(int h, int w, int quality, int sampling, uint8_t* out, int64_t cap) {
    int hs, vs;
    if (jpeg_enc_params(nullptr, quality, sampling, hs, vs)) return YF_ERR_ARG;
    if (!jpeg_enc_size_ok(h, w)) { set_err(nullptr, "size %dx%d outside [1, %d]", h, w, JPEG_MAX_SIDE); return YF_ERR_ARG; }
    if (!out || cap < JPEG_ENC_HEADER_BYTES) { set_err(nullptr, "the header takes %d bytes, cap is %lld", JPEG_ENC_HEADER_BYTES, (long long)cap); return YF_ERR_ARG; }
    return jpeg_enc_header(h, w, quality, hs, vs, out);
}

// every frame's size, its bytes against the frames buffer (frames_bytes >= 0) and, with out_off, its file against the output buffer
static int jpeg_enc_check(yf_ctx* ctx, int B, const int64_t* frame_off, const int32_t* h, const int32_t* w, int64_t frames_bytes, int hs,
                          int vs, const int64_t* out_off, int64_t out_bytes) {
    if (!frame_off || !h || !w) { set_err(&ctx->err, "null descriptor array"); return YF_ERR_ARG; }
    if (B < 1) { set_err(&ctx->err, "batch %d < 1", B); return YF_ERR_ARG; }
    for (int b = 0; b < B; ++b) {
        if (!jpeg_enc_size_ok(h[b], w[b])) { set_err(&ctx->err, "frame %d: size %dx%d outside [1, %d]", b, h[b], w[b], JPEG_MAX_SIDE); return YF_ERR_ARG; }
        const int64_t size = (int64_t)h[b] * w[b] * 3;
        if (frame_off[b] < 0 || (frames_bytes >= 0 && frame_off[b] > frames_bytes - size)) {
            set_err(&ctx->err, "frame %d: bytes [%lld, %lld) outside the %lld-byte buffer", b, (long long)frame_off[b],
                    (long long)(frame_off[b] + size), (long long)frames_bytes);
            return YF_ERR_ARG;
        }
        const int64_t bound = jpeg_enc_file_max(h[b], w[b], hs, vs);
        if (out_off && (out_off[b] < 0 || out_off[b] > out_bytes - bound)) {
            set_err(&ctx->err, "frame %d: file bytes [%lld, %lld) (yf_jpeg_encode_bound) outside the %lld-byte output buffer", b,
                    (long long)out_off[b], (long long)(out_off[b] + bound), (long long)out_bytes);
            return YF_ERR_ARG;
        }
    }
    return YF_OK;
}

static int jpeg_enc_grow(yf_ctx* ctx, unsigned char** p, size_t* cap, size_t need) {
    if (need <= *cap) return YF_OK;
    CU(cudaDeviceSynchronize());                        // an earlier call's kernels, on any stream, may still use the old buffer
    if (*p) CU(cudaFree(*p));
    *p = nullptr; *cap = 0;
    CU(cudaMalloc(p, need));
    *cap = need;
    return YF_OK;
}

// frames dev -> files at out + out_off[b], len dev [B]. Arguments already checked.
static int jpeg_enc_enqueue(yf_ctx* ctx, const uint8_t* frames, int B, const int64_t* frame_off, const int32_t* h, const int32_t* w,
                            int quality, int hs, int vs, uint8_t* out, const int64_t* out_off, int64_t* len, cudaStream_t st) {
    std::map<std::pair<int, int>, int32_t> hofs;        // one header per distinct size, all staged with one copy
    std::vector<uint8_t> hb;
    std::vector<JpegEncDesc> ds(B);
    for (int b = 0; b < B; ++b) {
        auto it = hofs.find({h[b], w[b]});
        if (it == hofs.end()) {
            it = hofs.emplace(std::make_pair(h[b], w[b]), (int32_t)hb.size()).first;
            hb.resize(hb.size() + JPEG_ENC_HEADER_BYTES);
            jpeg_enc_header(h[b], w[b], quality, hs, vs, hb.data() + it->second);
        }
        JpegEncDesc& d = ds[b];
        memset(&d, 0, sizeof d);
        d.src = frame_off[b]; d.dst = out_off[b];
        d.hdr = it->second; d.hdr_len = JPEG_ENC_HEADER_BYTES;
        d.h = (uint16_t)h[b]; d.w = (uint16_t)w[b]; d.hs = (uint8_t)hs; d.vs = (uint8_t)vs;
        d.mcux = (uint16_t)((w[b] + 8 * hs - 1) / (8 * hs)); d.mcuy = (uint16_t)((h[b] + 8 * vs - 1) / (8 * vs));
    }
    // workspace of the largest chunk: [coefficients, 128 B a block | bit offsets, 8 B a block | bit counts of the frames | bit buffers]
    int64_t most_blocks = 0, most_bits = 0;
    for (int c0 = 0; c0 < B; c0 += JPEG_ENC_CHUNK) {
        int64_t blocks = 0, bytes = 0;
        for (int i = c0; i < std::min(B, c0 + JPEG_ENC_CHUNK); ++i) {
            ds[i].cbase = blocks; ds[i].bbase = bytes;
            blocks += jpeg_enc_blocks(h[i], w[i], hs, vs);
            bytes += (jpeg_enc_scan_max(h[i], w[i], hs, vs) + 31) / 16 * 16;      // whole 16-byte loads of the stuffing stage
        }
        most_blocks = std::max(most_blocks, blocks);
        most_bits = std::max(most_bits, bytes);
    }
    // every part starts on a 256-byte boundary: the stuffing kernel reads the bit buffers with 16-byte loads
    auto up = [](size_t x) { return (x + 255) / 256 * 256; };
    const size_t off_offs = up((size_t)most_blocks * 128), off_fbits = up(off_offs + (size_t)most_blocks * 8);
    const size_t off_bits = up(off_fbits + sizeof(int64_t) * JPEG_ENC_CHUNK);
    int rc = jpeg_enc_grow(ctx, &ctx->d_jenc, &ctx->jenc_cap, off_bits + (size_t)most_bits);
    if (rc) return rc;
    if ((rc = jpeg_enc_grow(ctx, &ctx->d_jhdr, &ctx->jhdr_cap, hb.size()))) return rc;
    CU(cudaMemcpyAsync(ctx->d_jhdr, hb.data(), hb.size(), cudaMemcpyHostToDevice, st));
    int16_t* coef = reinterpret_cast<int16_t*>(ctx->d_jenc);
    int64_t* offs = reinterpret_cast<int64_t*>(ctx->d_jenc + off_offs);
    int64_t* fbits = reinterpret_cast<int64_t*>(ctx->d_jenc + off_fbits);
    uint8_t* bits = ctx->d_jenc + off_bits;
    JpegEncChunk ch;
    int qz[2][64];
    jpeg_enc_qtables(quality, qz);
    for (int t = 0; t < 2; ++t)
        for (int k = 0; k < 64; ++k) ch.qdiv[t][h_jpeg_natural[k]] = (uint16_t)(qz[t][k] << 3);
    for (int c0 = 0; c0 < B; c0 += JPEG_ENC_CHUNK) {
        const int n = std::min(JPEG_ENC_CHUNK, B - c0);
        int64_t max_blocks = 1;
        for (int i = 0; i < n; ++i) {
            ch.d[i] = ds[c0 + i];
            max_blocks = std::max(max_blocks, jpeg_enc_blocks(h[c0 + i], w[c0 + i], hs, vs));
        }
        constexpr int bpc = JPEG_ENC_DCT_NT / 8;           // 8x8 blocks per CTA and pass
        const dim3 gd((unsigned)std::min<int64_t>((max_blocks + bpc - 1) / bpc, 16384), (unsigned)n);
        jpeg_enc_dct_kernel<<<gd, JPEG_ENC_DCT_NT, 0, st>>>(frames, ch, coef);
        CU(cudaGetLastError());
        jpeg_enc_len_kernel<<<n, JPEG_ENC_SCAN_NT, 0, st>>>(ch, coef, offs, fbits, reinterpret_cast<uint32_t*>(bits));
        CU(cudaGetLastError());
        const dim3 ge((unsigned)std::min<int64_t>((max_blocks + JPEG_ENC_EMIT_NT - 1) / JPEG_ENC_EMIT_NT, 2048), (unsigned)n);
        jpeg_enc_emit_kernel<<<ge, JPEG_ENC_EMIT_NT, 0, st>>>(ch, coef, offs, fbits, reinterpret_cast<uint32_t*>(bits));
        CU(cudaGetLastError());
        jpeg_enc_stuff_kernel<<<n, JPEG_ENC_STUFF_NT, 0, st>>>(ch, ctx->d_jhdr, fbits, bits, out, len + c0);
        CU(cudaGetLastError());
        ctx->launches += 4;
    }
    return YF_OK;
}

extern "C" int yf_encode_jpeg(yf_ctx* ctx, const uint8_t* frames_dev, int B, const int64_t* frame_off, const int32_t* h, const int32_t* w,
                              int quality, int sampling, uint8_t* out_dev, const int64_t* out_off, int64_t out_bytes, int64_t* len_dev,
                              void* stream) {
    CTX_CHECK(ctx);
    if (!frames_dev || !out_dev || !out_off || !len_dev) { set_err(&ctx->err, "null frames, output, offset or length pointer"); return YF_ERR_ARG; }
    int hs, vs;
    int rc = jpeg_enc_params(&ctx->err, quality, sampling, hs, vs);
    if (rc || (rc = jpeg_enc_check(ctx, B, frame_off, h, w, -1, hs, vs, out_off, out_bytes))) return rc;
    CU(cudaSetDevice(ctx->device));
    return jpeg_enc_enqueue(ctx, frames_dev, B, frame_off, h, w, quality, hs, vs, out_dev, out_off, len_dev, (cudaStream_t)stream);
}

extern "C" int yf_encode_host_jpeg(yf_ctx* ctx, const uint8_t* frames_host, int64_t nbytes, int B, const int64_t* frame_off,
                                   const int32_t* h, const int32_t* w, int quality, int sampling, uint8_t* out_host, int64_t cap,
                                   int64_t* len_host, void* stream) {
    CTX_CHECK(ctx);
    cudaStream_t st = (cudaStream_t)stream;
    if (!frames_host || !out_host || !len_host) { set_err(&ctx->err, "null frames, output or length pointer"); return YF_ERR_ARG; }
    int hs, vs;
    int rc = jpeg_enc_params(&ctx->err, quality, sampling, hs, vs);
    if (rc || (rc = jpeg_enc_check(ctx, B, frame_off, h, w, nbytes, hs, vs, nullptr, 0))) return rc;
    std::vector<int64_t> staged(B);                     // each file at its bound on the device, then packed
    int64_t staged_bytes = 0;
    for (int b = 0; b < B; ++b) { staged[b] = staged_bytes; staged_bytes += jpeg_enc_file_max(h[b], w[b], hs, vs); }
    CU(cudaSetDevice(ctx->device));
    if ((rc = ensure_bgr(ctx, (size_t)nbytes, st))) return rc;
    if ((rc = jpeg_enc_grow(ctx, &ctx->d_jout, &ctx->jout_cap, (size_t)staged_bytes))) return rc;
    if ((rc = jpeg_enc_grow(ctx, reinterpret_cast<unsigned char**>(&ctx->d_jlen), &ctx->jlen_cap, sizeof(int64_t) * B))) return rc;
    CU(cudaMemcpyAsync(ctx->d_bgr, frames_host, (size_t)nbytes, cudaMemcpyHostToDevice, st));      // the frames, one copy
    if ((rc = jpeg_enc_enqueue(ctx, ctx->d_bgr, B, frame_off, h, w, quality, hs, vs, ctx->d_jout, staged.data(), ctx->d_jlen, st))) return rc;
    CU(cudaMemcpyAsync(len_host, ctx->d_jlen, sizeof(int64_t) * B, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    int64_t total = 0;
    for (int b = 0; b < B; ++b) total += len_host[b];
    if (total > cap) {
        set_err(&ctx->err, "the %d files take %lld bytes, out_host holds %lld", B, (long long)total, (long long)cap);
        return YF_ERR_ARG;
    }
    if ((rc = jpeg_enc_grow(ctx, &ctx->d_jpack, &ctx->jpack_cap, (size_t)std::max<int64_t>(total, 1)))) return rc;
    JpegPackChunk pk;
    int64_t pos = 0, most = 1;
    for (int c0 = 0; c0 < B; c0 += JPEG_ENC_CHUNK) {
        const int n = std::min(JPEG_ENC_CHUNK, B - c0);
        for (int i = 0; i < n; ++i) {
            pk.src[i] = staged[c0 + i]; pk.dst[i] = pos; pk.len[i] = len_host[c0 + i];
            pos += pk.len[i];
            most = std::max(most, pk.len[i]);
        }
        const dim3 gp((unsigned)std::min<int64_t>((most + 255) / 256, 1024), (unsigned)n);
        jpeg_enc_pack_kernel<<<gp, 256, 0, st>>>(pk, ctx->d_jout, ctx->d_jpack);
        CU(cudaGetLastError());
        ctx->launches += 1;
    }
    CU(cudaMemcpyAsync(out_host, ctx->d_jpack, (size_t)total, cudaMemcpyDeviceToHost, st));       // the files, one copy
    CU(cudaStreamSynchronize(st));
    return YF_OK;
}

// ---- asynchronous, double-buffered host path --------------------------------------------------------------
static int slots_init(yf_ctx* ctx) {
    if (ctx->s_copy) return YF_OK;
    CU(cudaStreamCreateWithFlags(&ctx->s_copy, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&ctx->s_comp, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&ctx->s_back, cudaStreamNonBlocking));
    const size_t npx = (size_t)ctx->max_batch * ctx->in_ch * ctx->H * ctx->W;
    for (int i = 0; i < 2; ++i) {
        CU(cudaMalloc(&ctx->sl_u8[i], npx));
        CU(cudaMalloc(&ctx->sl_counts[i], sizeof(int32_t) * ctx->max_batch));
        CU(cudaMalloc(&ctx->sl_status[i], sizeof(int32_t) * ctx->max_batch));
        CU(cudaEventCreateWithFlags(&ctx->sl_in[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ctx->sl_free[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ctx->sl_done[i], cudaEventDisableTiming));
    }
    return YF_OK;
}

static int submit_impl(yf_ctx* ctx, int slot, const uint8_t* u8_host, int B, const yf_post_params* p,
                       yf_det* out_host, int32_t* counts_host, int32_t* status_host, bool out_on_device);

extern "C" int yf_detect_submit_u8(yf_ctx* ctx, int slot, const uint8_t* u8_host, int B, const yf_post_params* p,
                                   yf_det* out_host, int32_t* counts_host, int32_t* status_host) {
    CTX_CHECK(ctx);
    return submit_impl(ctx, slot, u8_host, B, p, out_host, counts_host, status_host, false);
}

extern "C" int yf_detect_submit_u8_dev(yf_ctx* ctx, int slot, const uint8_t* u8_host, int B, const yf_post_params* p,
                                       yf_det* out_dev, int32_t* counts_dev, int32_t* status_dev) {
    CTX_CHECK(ctx);
    return submit_impl(ctx, slot, u8_host, B, p, out_dev, counts_dev, status_dev, true);
}

static int submit_impl(yf_ctx* ctx, int slot, const uint8_t* u8_host, int B, const yf_post_params* p,
                       yf_det* out_host, int32_t* counts_host, int32_t* status_host, bool out_on_device) {
    if (slot < 0 || slot > 1 || !u8_host || !p || !out_host || !counts_host) { set_err(&ctx->err, "bad argument"); return YF_ERR_ARG; }
    if (B < 1 || B > ctx->max_batch) { set_err(&ctx->err, "batch %d outside [1, max_batch=%d]", B, ctx->max_batch); return YF_ERR_STATE; }
    if (p->max_det < 1) { set_err(&ctx->err, "max_det must be >= 1"); return YF_ERR_ARG; }
    if (!ctx->weights_loaded) { set_err(&ctx->err, "yf_load_weights has not been called"); return YF_ERR_STATE; }
    CU(cudaSetDevice(ctx->device));
    int rc = slots_init(ctx);
    if (rc) return rc;
    if (p->max_det > ctx->sl_out_cap[slot]) {
        if (ctx->sl_used[slot]) CU(cudaEventSynchronize(ctx->sl_done[slot]));
        for (auto& kv : ctx->graphs) cudaGraphExecDestroy(kv.second.first);
        ctx->graphs.clear();
        if (ctx->sl_out[slot]) CU(cudaFree(ctx->sl_out[slot]));
        ctx->sl_out[slot] = nullptr;
        CU(cudaMalloc(&ctx->sl_out[slot], sizeof(yf_det) * (size_t)p->max_det * ctx->max_batch));
        ctx->sl_out_cap[slot] = p->max_det;
    }
    const size_t npx = (size_t)B * ctx->in_ch * ctx->H * ctx->W;
    if (ctx->sl_used[slot]) CU(cudaStreamWaitEvent(ctx->s_copy, ctx->sl_free[slot], 0));   // previous batch of this slot has been consumed
    CU(cudaMemcpyAsync(ctx->sl_u8[slot], u8_host, npx, cudaMemcpyHostToDevice, ctx->s_copy));
    CU(cudaEventRecord(ctx->sl_in[slot], ctx->s_copy));
    CU(cudaStreamWaitEvent(ctx->s_comp, ctx->sl_in[slot], 0));
    if (ctx->sl_used[slot]) CU(cudaStreamWaitEvent(ctx->s_comp, ctx->sl_done[slot], 0));   // the slot's previous results have left its buffers
    if (out_on_device) {    // results go straight into the caller's device buffers (e.g. to be gathered with NCCL)
        rc = detect_impl(ctx, ctx->sl_u8[slot], true, B, p, out_host, counts_host, status_host ? status_host : ctx->sl_status[slot], ctx->s_comp);
        if (rc) return rc;
        CU(cudaEventRecord(ctx->sl_free[slot], ctx->s_comp));
    } else {
        rc = detect_fixed(ctx, ctx->sl_u8[slot], true, B, p, ctx->sl_out[slot], ctx->sl_counts[slot], ctx->sl_status[slot], ctx->s_comp);
        if (rc) return rc;
        CU(cudaEventRecord(ctx->sl_free[slot], ctx->s_comp));
        // the results travel back on their own stream, so the next batch's kernels start right behind this batch's
        CU(cudaStreamWaitEvent(ctx->s_back, ctx->sl_free[slot], 0));
        CU(cudaMemcpyAsync(out_host, ctx->sl_out[slot], sizeof(yf_det) * (size_t)B * p->max_det, cudaMemcpyDeviceToHost, ctx->s_back));
        CU(cudaMemcpyAsync(counts_host, ctx->sl_counts[slot], sizeof(int32_t) * B, cudaMemcpyDeviceToHost, ctx->s_back));
        if (status_host) CU(cudaMemcpyAsync(status_host, ctx->sl_status[slot], sizeof(int32_t) * B, cudaMemcpyDeviceToHost, ctx->s_back));
    }
    CU(cudaEventRecord(ctx->sl_done[slot], out_on_device ? ctx->s_comp : ctx->s_back));
    ctx->sl_used[slot] = true;
    return YF_OK;
}

extern "C" int yf_detect_wait(yf_ctx* ctx, int slot) {
    CTX_CHECK(ctx);
    if (slot < 0 || slot > 1 || !ctx->sl_used[slot]) { set_err(&ctx->err, "slot %d has no submitted batch", slot); return YF_ERR_STATE; }
    CU(cudaEventSynchronize(ctx->sl_done[slot]));
    return YF_OK;
}

extern "C" int yf_compact_dets(yf_ctx* ctx, const yf_det* dets, const int32_t* counts, int B, int max_det, void* packed, int hdr_slots,
                               int cap_records, void* stream) {
    CTX_CHECK(ctx);
    if (!dets || !counts || !packed || B < 1 || max_det < 1 || hdr_slots < B + 2 || cap_records < 0) { set_err(&ctx->err, "bad argument"); return YF_ERR_ARG; }
    if (hdr_slots % 2) { set_err(&ctx->err, "hdr_slots must be even (records are 8-byte aligned)"); return YF_ERR_ARG; }
    int32_t* hdr = reinterpret_cast<int32_t*>(packed);
    compact_dets_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(dets, counts, B, max_det, hdr, hdr_slots, reinterpret_cast<yf_det*>(hdr + hdr_slots), cap_records);
    ctx->launches++;
    CU(cudaGetLastError());
    return YF_OK;
}

extern "C" int64_t yf_launch_count(const yf_ctx* ctx) { return ctx ? ctx->launches : -1; }
