/*
 * yf.h — C ABI of the B200-native YOLO-Fastest detection hot path (libyf_b200.so).
 *
 * The reference (JunFenngZhi/YOLO-Fastest-and-Embedded-deployment) has no FFI/plugin interface:
 * its boundary for this path is a Python object API (SURVEY.md §8b).  Each entry point below
 * replaces one piece of that API; the Python host shim in yolo_fastest_b200/ keeps the
 * reference's class names and signatures and calls these through ctypes.  Citations are
 * relative to the reference repo root.
 *
 * Conventions
 *   - every call returns 0 on success or a negative yf_status; nothing throws across the ABI;
 *     yf_last_error() gives the message of the last failure (per ctx, or global when ctx==NULL)
 *   - "dev" pointers are caller-owned CUDA device memory on the ctx's device, "host" pointers
 *     are ordinary host memory; the library owns only its packed weights and workspaces
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy default
 *     stream); only the *_host entry points synchronise
 *   - a ctx is bound to one device, is NOT thread-safe, and is sized at creation
 *   - tensors are fp32, NCHW, contiguous — the reference's own layout
 *     (src/model_training/model/yolo_fastest.py:150-218)
 *   - there is no CPU fallback: without a CUDA device every compute call fails with YF_ERR_CUDA
 */
#ifndef YF_B200_H
#define YF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YF_ABI_VERSION 1
#define YF_MAX_ANCHORS 8

typedef enum {
    YF_OK = 0,
    YF_ERR_ARG = -1,      /* bad argument / unsupported configuration */
    YF_ERR_CUDA = -2,     /* CUDA runtime error (message has the cudaError string) */
    YF_ERR_STATE = -3,    /* call order: weights not loaded, batch > max_batch, ... */
    YF_ERR_DOMAIN = -4    /* input outside the reference's defined domain (see yf_postprocess) */
} yf_status;

typedef struct yf_ctx yf_ctx; /* opaque */

/* One detection.  Row layout of the reference's result lists
 *   detect flavour  [x1, y1, x2, y2, conf, cls_score, cls_index]  (src/detect.py:65-66)
 *   validate flavour (x1, y1, x2, y2, obj_conf, class_conf, class_pred) (src/model_training/utils/general.py:111)
 * plus `src` = index of the candidate in decode order (head_large first, then anchor, row, col —
 * src/detect.py:43,54-56), which the reference does not return but which makes orders testable.
 * detect flavour: coordinates are integers (Python round(), half-to-even) held exactly in doubles,
 * conf/cls_score are the float64 sigmoids.  validate flavour: every field is the fp32 value widened. */
typedef struct {
    double x1, y1, x2, y2;
    double conf, cls_score;
    int32_t cls;
    int32_t src;
} yf_det; /* 56 bytes */

/* Model variants (SURVEY 8f-4). YF_VARIANT_LITE = the reference's YoloFastest_lite (yolo_fastest.py:234-372): the same parameter set
 * with heads of (num_anchors * num_cls) * (5 + num_cls) channels (:240-241), a forward that goes conv3_2 -> conv3_4 without the depthwise
 * conv3_3 (:335-337) and ends at head_5 (:365-372): yf_forward then writes head_small only (head_large may be NULL). */
enum { YF_VARIANT_FULL = 0, YF_VARIANT_LITE = 1 };

enum { YF_MODE_DETECT = 0,   /* src/detect.py:41-84,155-169 */
       YF_MODE_VALIDATE = 1  /* src/model_training/loss/yolo_loss.py:98-141 + utils/general.py:87-143 */ };

/* ---- lifecycle -------------------------------------------------------------------------- */

/* Replaces YoloFastest(io_params).to(device) (yolo_fastest.py:70-148; detect.py:89).
 * in_ch is 1 (io_params["input_channel"], _config.py:10: the shipped models) or 3 (colour input, yolo_fastest.py:73,78: planes
 * in the order the reference feeds them, i.e. R, G, B after detect.py:121); H and W multiples of 32
 * (_config.py:11).  Head shapes follow: large = [B, A*(5+nc), H/16, W/16], small = [.., H/32, W/32]. */
int yf_create(yf_ctx** out, int device, int in_ch, int num_cls, int num_anchors,
              int max_batch, int H, int W);
/* The same for a model variant: YF_VARIANT_FULL == yf_create; YF_VARIANT_LITE replaces YoloFastest_lite(io_params)
 * (yolo_fastest.py:234-319), single-channel input. */
int yf_create_variant(yf_ctx** out, int device, int in_ch, int num_cls, int num_anchors,
                      int max_batch, int H, int W, int variant);
void yf_destroy(yf_ctx* ctx);
const char* yf_last_error(const yf_ctx* ctx);
int yf_abi_version(void);

/* Number of floats yf_load_weights expects for this architecture (host-side helper, no CUDA). */
int64_t yf_weight_count(int in_ch, int num_cls, int num_anchors);
int64_t yf_weight_count_variant(int in_ch, int num_cls, int num_anchors, int variant);

/* Replaces model.load_state_dict(torch.load(path)) + .eval() (detect.py:89-91).
 * `host_blob`: BatchNorm-folded fp32 parameters in forward order, per conv its weight in PyTorch
 * layout ([Cout][Cin/groups][k][k]; ConvTranspose2d: [Cin][Cout][2][2]) followed by its bias
 * [Cout] — 86 convs, yolo_fastest.py:78-148.  Copied; the caller keeps ownership. Synchronous. */
int yf_load_weights(yf_ctx* ctx, const float* host_blob, int64_t n_floats);

/* ---- forward ---------------------------------------------------------------------------- */

/* Replaces YoloFastest.forward (yolo_fastest.py:150-218): x dev [B, in_ch, H, W] ->
 * head_large dev [B, A*(5+nc), H/16, W/16], head_small dev [B, A*(5+nc), H/32, W/32]. B <= max_batch. */
int yf_forward(yf_ctx* ctx, const float* x, int B, float* head_large, float* head_small, void* stream);

/* Debug/parity tap: copies the named intermediate activation of the LAST yf_forward (NCHW fp32,
 * name = the reference attribute producing it, e.g. "res2_1", "conv4_2", "conv5_2", "conv4_1_1")
 * into dst (dev). Returns the number of floats per image through *per_image (may be called with
 * dst == NULL to query). Only group outputs exist as tensors; fused intermediates do not. */
int yf_tap(yf_ctx* ctx, const char* name, int B, float* dst, int64_t* per_image, void* stream);

/* ---- post-processing -------------------------------------------------------------------- */

/* Post-processing parameters = YOLO_post_process.__init__ (detect.py:15-21) /
 * YOLOLossV3.__init__ + non_max_suppression args (yolo_loss.py:28-36, general.py:87). */
typedef struct {
    double anchors[2][YF_MAX_ANCHORS][2]; /* [head(large,small)][anchor][w,h] in input pixels (_config.py:5-9) */
    double conf_thres;                    /* detect: keep conf >  thres (detect.py:58); validate: >= (general.py:100) */
    double nms_thres;                     /* detect: drop IoU  >  thres (detect.py:79); validate: keep IoU < thres (general.py:136) */
    int32_t input_h, input_w;             /* io_params["input_shape"][0:2] */
    int32_t mode;                         /* YF_MODE_DETECT | YF_MODE_VALIDATE */
    int32_t max_det;                      /* capacity of out per image */
} yf_post_params;

/* Replaces decode_box + class split + stable sort + non_maxium_supression for a whole batch
 * (detect.py:41-84,155-169), or YOLOLossV3(targets=None) + cat + non_max_suppression
 * (validate.py:38-44) in YF_MODE_VALIDATE.
 * heads: dev, shapes as produced by yf_forward for (hl, wl) = large map, (hs, ws) = small map.
 * out: dev [B][max_det] in the reference's output order (class ascending, conf descending,
 * ties in candidate order); counts: dev [B] = number kept (if > max_det the list was truncated).
 * status (dev int32[B], may be NULL): bit0 = a coordinate magnitude exceeded 2^25 (areas no
 * longer exact in fp64; the reference uses big ints there), bit1 = a non-finite logit was seen. */
int yf_postprocess(yf_ctx* ctx, const float* head_large, const float* head_small, int B,
                   int hl, int wl, int hs, int ws, const yf_post_params* p,
                   yf_det* out, int32_t* counts, int32_t* status, void* stream);

/* Decode only, no NMS: every candidate with conf > conf_thres in decode order — the list
 * YOLO_post_process.decode_box returns (detect.py:41-67), for each image of the batch. */
int yf_decode(yf_ctx* ctx, const float* head_large, const float* head_small, int B,
              int hl, int wl, int hs, int ws, const yf_post_params* p,
              yf_det* out, int32_t* counts, int32_t* status, void* stream);

/* Replaces YOLOLossV3.forward(input, targets=None) for one head (yolo_loss.py:48-68,98-141):
 * head dev [B, A*(5+nc), h, w] -> out dev [B, A*h*w, 5+nc] fp32, rows (anchor,row,col),
 * columns (cx, cy, w, h, conf, cls...). anchors: host [A][2]. */
int yf_val_decode(yf_ctx* ctx, const float* head, int B, int h, int w, const double* anchors,
                  int num_anchors, int num_cls, int input_h, int input_w, float* out, void* stream);

/* Replaces non_max_suppression(prediction, num_classes, conf_thres, nms_thres) (general.py:87-143) for
 * callers that hold the decoded tensor: pred dev [B][N][5+nc] fp32, rows (cx, cy, w, h, conf, cls...)
 * as YOLOLossV3 / yf_val_decode produce and validate.py:42 concatenates. Output as yf_postprocess in
 * YF_MODE_VALIDATE; N must not exceed the ctx's candidate capacity. pred is not modified (the
 * reference overwrites its xywh with xyxy, general.py:95). */
int yf_val_nms(yf_ctx* ctx, const float* pred, int B, int N, double conf_thres, double nms_thres,
               int max_det, yf_det* out, int32_t* counts, int32_t* status, void* stream);

/* NMS on caller-supplied boxes — the bit-exactness test entry.
 * YF_MODE_DETECT: YOLO_post_process.non_maxium_supression (detect.py:69-84) on a list already
 *   sorted by conf descending; boxes dev [n][4] int32 (x1,y1,x2,y2); keep dev [n] receives the
 *   indices of kept boxes in order; *n_keep (dev) their number.
 * YF_MODE_VALIDATE: the per-class loop of non_max_suppression (general.py:121-136) with bbox_iou
 *   (+1 convention, general.py:29-52); boxes_f dev [n][4] fp32 sorted by conf descending. */
int yf_nms_sorted_i32(yf_ctx* ctx, const int32_t* boxes, int n, double nms_thres,
                      int32_t* keep, int32_t* n_keep, void* stream);
int yf_nms_sorted_f32(yf_ctx* ctx, const float* boxes_f, int n, float nms_thres,
                      int32_t* keep, int32_t* n_keep, void* stream);

/* ---- fused paths ------------------------------------------------------------------------ */

/* forward + postprocess with heads kept in the library's workspace: the batched equivalent of
 * the body of Detect_YOLO.batch_detect (detect.py:152-169). x dev [B, in_ch, H, W]. */
int yf_detect(yf_ctx* ctx, const float* x, int B, const yf_post_params* p,
              yf_det* out, int32_t* counts, int32_t* status, void* stream);

/* Same through HOST buffers (the end-to-end call): copies x_host [B, in_ch, H, W] fp32 to the
 * device, runs yf_detect, copies out/counts/status back and synchronises `stream`.
 * Pinned host memory makes the copies asynchronous; pageable memory works too. */
int yf_detect_host(yf_ctx* ctx, const float* x_host, int B, const yf_post_params* p,
                   yf_det* out_host, int32_t* counts_host, int32_t* status_host, void* stream);

/* Same with the numeric tail of Detect_YOLO.__pre_process fused in (detect.py:123-124):
 * u8_host [B, H, W] grayscale uint8 -> (x - 128) / 255 on the device. */
int yf_detect_host_u8(yf_ctx* ctx, const uint8_t* u8_host, int B, const yf_post_params* p,
                      yf_det* out_host, int32_t* counts_host, int32_t* status_host, void* stream);

/* Asynchronous, double-buffered form of yf_detect_host_u8 for serving loops: two slots (0, 1), each with its own
 * device staging and result buffers. yf_detect_submit_u8 enqueues the H2D copy on an internal copy stream and
 * the detection + D2H of the results on an internal compute stream and returns immediately; yf_detect_wait
 * blocks until the slot's results are in out_host / counts_host / status_host. Submitting batch i+1 into the
 * other slot before waiting for batch i overlaps its H2D copy with the compute of batch i. The host buffers
 * must stay valid (and should be pinned) until the wait returns. */
int yf_detect_submit_u8(yf_ctx* ctx, int slot, const uint8_t* u8_host, int B, const yf_post_params* p,
                        yf_det* out_host, int32_t* counts_host, int32_t* status_host);
int yf_detect_wait(yf_ctx* ctx, int slot);
/* Same submission with the results left in caller-owned DEVICE buffers (out_dev [B][max_det], counts_dev [B],
 * status_dev [B] or NULL) — for multi-GPU jobs that return their slabs to rank 0 with a collective. After
 * yf_detect_wait the buffers are complete and may be read from any stream. */
int yf_detect_submit_u8_dev(yf_ctx* ctx, int slot, const uint8_t* u8_host, int B, const yf_post_params* p,
                            yf_det* out_dev, int32_t* counts_dev, int32_t* status_dev);

/* ---- multi-GPU result return (SURVEY 8e) ------------------------------------------------------ */

/* Compacts the per-image slabs of yf_detect / yf_detect_submit_u8_dev (dets dev [B][max_det], counts dev [B]) into ONE contiguous
 * message: packed dev = int32 header [total, B, n_0 .. n_{B-1}] in `hdr_slots` int32 words (even, >= B + 2), followed by the records of
 * image 0, 1, ... back to back, n_b = min(counts[b], max_det), at most cap_records of them; `total` is the untruncated sum, so a
 * receiver sees an overflow instead of a silent cut. The reference is single-process (SURVEY 2.1); this is the payload of the one
 * collective that returns per-rank detection lists to rank 0 (yolo_fastest_b200/dist.py). */
int yf_compact_dets(yf_ctx* ctx, const yf_det* dets, const int32_t* counts, int B, int max_det, void* packed, int hdr_slots,
                    int cap_records, void* stream);

/* ---- pre-processing on the device (SURVEY 8f-1) ------------------------------------------ */

/* Replaces the image half of Detect_YOLO.__pre_process (detect.py:107-122): cv2.cvtColor(BGR2GRAY) followed by
 * cv2.resize(img, (W, H)) (INTER_LINEAR) for a batch of frames as cv2.imread returns them.
 * bgr dev [B, Ho, Wo, 3] uint8 (interleaved B, G, R) -> gray dev [B, H, W] uint8, H and W those of yf_create.
 * Integer arithmetic identical to OpenCV 4.x for 8-bit images, so the bytes equal the host path's; with
 * Ho == H and Wo == W the resize is the identity, as in the reference, which then skips it. The normalisation
 * (x - 128) / 255 (detect.py:124) stays fused into the first convolution of the u8 entry points. */
int yf_preprocess_bgr(yf_ctx* ctx, const uint8_t* bgr, int B, int Ho, int Wo, uint8_t* gray, void* stream);

/* yf_detect_host_u8 with that pre-processing in front: bgr_host [B, Ho, Wo, 3] uint8 host frames -> detections in
 * NETWORK-input coordinates (Detect_YOLO.__adjust_coord, detect.py:131-139, stays with the caller). */
int yf_detect_host_bgr(yf_ctx* ctx, const uint8_t* bgr_host, int B, int Ho, int Wo, const yf_post_params* p,
                       yf_det* out_host, int32_t* counts_host, int32_t* status_host, void* stream);

/* The same for a batch whose frames may differ in size, and for colour networks: frames dev holds B BGR uint8 frames back to back,
 * frame b at byte offset off[b] with shape [Ho[b], Wo[b], 3] and contiguous rows, 1 <= Ho[b], Wo[b] <= 16384. off / Ho / Wo are
 * HOST arrays, B <= max_batch. out dev: [B, H, W] gray when in_ch == 1 (the bytes of yf_preprocess_bgr), [B, 3, H, W] R, G, B planes
 * when in_ch == 3 (detect.py:107-122 for a colour network: cv2.resize of the BGR frame, then [:, :, ::-1] and HWC -> CHW; the 11-bit
 * arithmetic of the gray path once per channel). The coefficients are computed on the device for each frame, so sizes may change from
 * call to call, and within a call, without a synchronisation. Frames whose rows are 4-byte aligned (width a multiple of 4, aligned
 * offset) are read fastest; any layout works. Bad descriptors fail with YF_ERR_ARG before anything is enqueued. */
int yf_preprocess_frames(yf_ctx* ctx, const uint8_t* frames, int B, const int64_t* off, const int32_t* Ho, const int32_t* Wo,
                         uint8_t* out, void* stream);

/* yf_detect_host_bgr for such a batch: frames_host holds the packed frames in `nbytes` bytes of HOST memory (pinned for an
 * asynchronous copy; every descriptor must lie inside them). One copy of the nbytes to the device, yf_preprocess_frames, yf_detect,
 * and the results back as yf_detect_host_u8 returns them, in NETWORK-input coordinates (scaling back to each frame stays with the
 * caller). Synchronises `stream`. */
int yf_detect_host_frames(yf_ctx* ctx, const uint8_t* frames_host, int64_t nbytes, int B, const int64_t* off, const int32_t* Ho,
                          const int32_t* Wo, const yf_post_params* p, yf_det* out_host, int32_t* counts_host,
                          int32_t* status_host, void* stream);

/* ---- baseline JPEG files decoded on the device --------------------------------------------------------------------------- */

/* Status bit of yf_decode_jpeg / yf_detect_host_jpeg: the file's entropy-coded data ended early, held an invalid Huffman code, or
 * missed or misordered an RSTn marker (libjpeg warns and pads with zeros there; the device output of such a file is not cv2's). */
#define YF_STATUS_JPEG_CORRUPT 4

/* Host only, no CUDA: 0 and the decoded size if the device decoder takes this file, else YF_ERR_ARG with the reason in
 * yf_last_error(NULL). Taken: baseline sequential Huffman-coded files (SOF0, SOF1) with 8-bit samples and one interleaved scan of
 * every component; gray, or YCbCr at 4:4:4, 4:2:2 or 4:2:0; restart intervals; files without DHT segments (the T.81 K.3 tables);
 * sizes 1 .. 16384. Turned down: progressive, arithmetic, lossless and hierarchical files, 12-bit samples, 2 or 4 components,
 * other sampling factors, several scans, RGB files (Adobe transform 0, or component IDs R, G, B without JFIF / Adobe markers),
 * EXIF orientations other than 1 (cv2 rotates those), truncated or malformed headers, and bytes that are not a JPEG. */
int yf_jpeg_probe(const uint8_t* data, int64_t nbytes, int32_t* h, int32_t* w);

/* B JPEG files back to back in HOST memory (file b = bytes [off[b], off[b] + len[b]) of files_host, nbytes in all) ->
 * the BGR frames cv2.imdecode(IMREAD_COLOR) returns, byte for byte, at frame_off[b] of frames_dev (frames_bytes long; [h, w, 3],
 * contiguous rows: the layout yf_preprocess_frames reads). status_dev [B]: YF_STATUS_JPEG_CORRUPT. off / len / frame_off are HOST
 * arrays. Every header is parsed and checked before anything is enqueued; one copy of the nbytes, then 3 kernel launches per 256
 * files. The decoder reads no byte of a file outside its [off[b], off[b] + len[b]).
 * Enqueued on `stream`; files_host must stay unchanged until the stream has passed the call. */
int yf_decode_jpeg(yf_ctx* ctx, const uint8_t* files_host, int64_t nbytes, int B, const int64_t* off, const int64_t* len,
                   uint8_t* frames_dev, const int64_t* frame_off, int64_t frames_bytes, int32_t* status_dev, void* stream);

/* yf_detect_host_frames for JPEG files: one copy of the files, decode, yf_preprocess_frames, yf_detect, results back in
 * NETWORK-input coordinates; status_host also carries bit 2 (when status_host is NULL a corrupt file fails the call with
 * YF_ERR_DOMAIN). frames_host (may be NULL) receives the decoded frames at frame_off, for callers that draw on them.
 * B <= max_batch. Synchronises `stream`. */
int yf_detect_host_jpeg(yf_ctx* ctx, const uint8_t* files_host, int64_t nbytes, int B, const int64_t* off, const int64_t* len,
                        const int64_t* frame_off, const yf_post_params* p, yf_det* out_host, int32_t* counts_host,
                        int32_t* status_host, uint8_t* frames_host, void* stream);

/* ---- baseline JPEG files encoded on the device -------------------------------------------------------------------------- */

/* Chroma sampling of the encoder, with the values of cv2.IMWRITE_JPEG_SAMPLING_FACTOR_* so that callers can pass those through. */
#define YF_JPEG_SAMPLING_420 0x221111   /* = cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2's default */
#define YF_JPEG_SAMPLING_422 0x211111
#define YF_JPEG_SAMPLING_444 0x111111

/* Host only, no CUDA: the most bytes one encoded file of an h x w frame can take (headers, every scan byte stuffed, EOI), or
 * YF_ERR_ARG (size outside [1, 16384], other sampling factors) with the reason in yf_last_error(NULL). */
int64_t yf_jpeg_encode_bound(int h, int w, int sampling);
/* Host only: the header bytes (SOI .. SOS) cv2.imencode writes for these parameters into out (cap bytes); returns their length (623)
 * or YF_ERR_ARG (quality outside [1, 100], other sampling factors, size outside [1, 16384], cap too small). */
int yf_jpeg_encode_header(int h, int w, int quality, int sampling, uint8_t* out, int64_t cap);
/* B BGR uint8 frames in DEVICE memory (frame b at byte offset frame_off[b] of frames_dev, [h[b], w[b], 3], contiguous rows: the layout
 * yf_decode_jpeg writes and yf_preprocess_frames reads) -> B JPEG files, each byte for byte what
 * cv2.imencode(".jpg", frame, [IMWRITE_JPEG_QUALITY, quality, IMWRITE_JPEG_SAMPLING_FACTOR, sampling]) returns: baseline, standard
 * Huffman tables, no restart intervals, JFIF APP0. File b goes to out_dev + out_off[b], which must have room for
 * yf_jpeg_encode_bound bytes inside the out_bytes of out_dev; len_dev [B] int64 (device) receives the length of each file.
 * frame_off / h / w / out_off are HOST arrays; every argument is checked before anything is enqueued. 4 kernel launches per 256
 * frames. Enqueued on `stream`. The frames are BGR [h, w, 3] by construction, and the entry points have no parameter for restart
 * intervals, optimised or progressive coding or a separate chroma quality: those outputs are not produced. */
int yf_encode_jpeg(yf_ctx* ctx, const uint8_t* frames_dev, int B, const int64_t* frame_off, const int32_t* h, const int32_t* w,
                   int quality, int sampling, uint8_t* out_dev, const int64_t* out_off, int64_t out_bytes, int64_t* len_dev,
                   void* stream);
/* The same from HOST frames (frames_host, nbytes long; every frame must lie inside): one copy of the nbytes to the device, the encode,
 * the lengths back into len_host [B], then ONE copy of the files packed back to back (file b right after file b - 1) into out_host.
 * When the files take more than `cap` bytes the call fails with YF_ERR_ARG naming the need, len_host holds the lengths, and nothing is
 * written to out_host. Synchronises `stream`. */
int yf_encode_host_jpeg(yf_ctx* ctx, const uint8_t* frames_host, int64_t nbytes, int B, const int64_t* frame_off,
                        const int32_t* h, const int32_t* w, int quality, int sampling, uint8_t* out_host, int64_t cap,
                        int64_t* len_host, void* stream);

/* ---- YUV 4:2:0 video frames (NV12, I420) on the device -------------------------------------------------------------------- */

/* One 8-bit YUV 4:2:0 frame of h x w pixels, h and w even, every plane at a byte offset from one base pointer. Luma row r is the w bytes
 * at y_off + r * y_pitch. Chroma sample k (0 <= k < w / 2) of chroma row r (0 <= r < h / 2) is at u_off + r * c_pitch + k * c_step,
 * and likewise from v_off. Pixel (r, c) takes chroma sample c / 2 of chroma row r / 2.
 *   NV12 (hardware decoders): c_step = 2, v_off = u_off + 1, the interleaved UV plane after a luma plane of the surface's height.
 *   I420 (yuv420p, FFmpeg, software decoders): c_step = 1, three separate planes (cv2's [3h/2, w] layout: u_off = h * w,
 *   v_off = u_off + (h / 2) * (w / 2), c_pitch = w / 2).
 * 48 bytes (4 bytes of tail padding). */
typedef struct {
    int64_t y_off, u_off, v_off;
    int32_t y_pitch, c_pitch, c_step;
    int32_t h, w;
} yf_yuv420;

/* The three YUV entry points check every descriptor before anything is enqueued, and fail with YF_ERR_ARG and a reason that names the
 * frame: h and w even and in [2, 16384]; y_pitch >= w; c_step >= 1; c_pitch >= (w / 2) * c_step; every byte of every plane inside
 * [base_dev, base_dev + nbytes); 1 <= B <= max_batch. desc_host is a HOST array of B descriptors. The arithmetic is cv2's for
 * COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420 (BT.601, limited range, 20-bit fixed point), whatever the layout.
 *
 * B frames -> the BGR frames cv2.cvtColor returns, byte for byte, at frame_off[b] of frames_dev ([h, w, 3], contiguous rows: the layout
 * yf_preprocess_frames reads and yf_encode_jpeg takes; frame_off is a HOST array, every frame inside the frames_bytes of frames_dev).
 * One launch per 256 frames, enqueued on `stream`. */
/* Host only, no CUDA: those descriptor checks without a ctx (no max_batch bound); 0, or YF_ERR_ARG with the reason in
 * yf_last_error(NULL). */
int yf_yuv420_check(int64_t nbytes, int B, const yf_yuv420* desc_host);
int yf_yuv420_to_bgr(yf_ctx* ctx, const uint8_t* base_dev, int64_t nbytes, int B, const yf_yuv420* desc_host, uint8_t* frames_dev,
                     const int64_t* frame_off, int64_t frames_bytes, void* stream);
/* B frames -> out dev as yf_preprocess_frames writes it for the BGR frames of yf_yuv420_to_bgr ([B, H, W] gray, or [B, 3, H, W] R, G, B
 * planes for in_ch == 3), byte for byte, without writing the BGR frames anywhere. One launch per 256 frames, enqueued on `stream`. */
int yf_preprocess_yuv420(yf_ctx* ctx, const uint8_t* base_dev, int64_t nbytes, int B, const yf_yuv420* desc_host, uint8_t* out_dev,
                         void* stream);
/* yf_preprocess_yuv420 into the ctx's own input buffer, then yf_detect's forward, decode and NMS: out_dev [B][max_det], counts_dev [B]
 * and status_dev [B] (may be NULL) as yf_detect writes them, in NETWORK-input coordinates. Enqueued on `stream` without a
 * synchronisation, after the asynchronous slots in flight. */
int yf_detect_yuv420(yf_ctx* ctx, const uint8_t* base_dev, int64_t nbytes, int B, const yf_yuv420* desc_host, const yf_post_params* p,
                     yf_det* out_dev, int32_t* counts_dev, int32_t* status_dev, void* stream);

/* ---- introspection ---------------------------------------------------------------------- */

/* Kernels launched by this ctx since creation (the bench's gpu_launches evidence). */
int64_t yf_launch_count(const yf_ctx* ctx);
/* Per-group device time of one forward at batch B (debug/profiling aid; synchronises).
 * names[i] points at static strings; ms[i] = milliseconds of group i. Returns number of groups
 * written (<= cap) or a negative status. */
int yf_profile_forward(yf_ctx* ctx, const float* x, int B, const char** names, float* ms, int cap);

#ifdef __cplusplus
}
#endif
#endif /* YF_B200_H */
