/*
 * yolo_b200.h — C-ABI of the B200-native fixed-point slim_yolo_v2 forward pass.
 *
 * This is the drop-in boundary for ONE hot path of
 * ZLkanyo009/Yolo-compression-and-deployment-in-FPGA: the BN-fused 8-bit
 * fixed-point slim_yolo_v2 forward that c_embedding/yolo_forward.c drives on the
 * FPGA accelerator and models/slim_yolo_v2.py simulates
 * (SlimYOLOv2_quantize_bnfuse).  Plain pointers and sizes only; no torch types.
 *
 * Each entry point cites the reference interface it replaces
 * (paths relative to the reference checkout).
 *
 * Data layouts (all int8 feature maps are NHWC, channel stride padded):
 *   - network input, int8:  [n][h][w][4]   = (R,G,B,0), the word the C driver
 *     packs per pixel (yolo_forward.c:95-96,116)
 *   - network input, RGB444: uint16 [n][h][w], 0x0BGR (ov7670.h:203-230,
 *     yolo_forward.c:57-85)
 *   - network input, fp32:  [n][3][h][w] RGB, ImageNet-normalised (test.py:79-80)
 *   - layer l output: int8 [n][h'][w'][cs], cs = yolo_b200_cstride(cout)
 *     = cout rounded up to a multiple of 16 (35 -> 48), pad channels are 0.
 *   - weights: int8, one of the YOLO_B200_WLAYOUT_* layouts; biases int8 [cout].
 *
 * Return codes: 0 = ok, negative = error (see yolo_b200_last_error()).
 */
#ifndef YOLO_B200_H
#define YOLO_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YOLO_B200_MAX_LAYERS   32
#define YOLO_B200_MAX_ANCHORS  8

/* Arithmetic contracts (SURVEY.md section 8a). */
#define YOLO_B200_CONTRACT_F   0  /* "FPGA": 3-shift programme of set_quantize_scale, yolo_forward.c:233-257 */
#define YOLO_B200_CONTRACT_P   1  /* PyTorch fake-quant: single RNE per layer, slim_yolo_v2.py:16-38,212-328 */

/* Rounding of right shifts in contract F (the RTL is absent; parameter). */
#define YOLO_B200_ROUND_RNE      0
#define YOLO_B200_ROUND_FLOOR    1
#define YOLO_B200_ROUND_HALF_UP  2

/* Weight layouts accepted by yolo_b200_load(). */
#define YOLO_B200_WLAYOUT_OIHW     0  /* PyTorch conv weight [cout][cin][3][3]  (slim_yolo_v2.py:59-87) */
#define YOLO_B200_WLAYOUT_OHWI     1  /* [cout][kh][kw][cin] */
#define YOLO_B200_WLAYOUT_WEIGHT_H 2  /* weight.h burst order [kh][kw][cout/Tm][cin/Tn][Tm][Tn], Tm=32,Tn=16
                                         (inferred from load_weight, yolo_forward.c:165-173,696-701) */

/* Detection-head semantics. */
#define YOLO_B200_HEAD_PYTHON  0  /* slim_yolo_v2.py:330-358,111-210: sigmoid/softmax, boxes normalised to [0,1],
                                     score >= conf_thresh, per-class greedy NMS (ovr <= thresh keeps), output in
                                     ascending anchor-index order */
#define YOLO_B200_HEAD_C       1  /* yolo_forward.c:965-1147 restated on its well-defined subset: sigma(-x) as
                                     written (:965-968), 2-way softmax, score > conf_thresh, h decoded with the
                                     anchor WIDTH (:1044), integer-pixel boxes, class-agnostic NMS suppressing
                                     iou >= thresh (:1128-1147), output in descending-score order */

typedef struct yolo_b200_layer {
    int32_t cin;    /* logical input channels  */
    int32_t cout;   /* logical output channels */
    int32_t activ;  /* 1 = leaky-ReLU slope 1/8 (utils/modules.py:25)      */
    int32_t pool;   /* 1 = 2x2 stride-2 max-pool after the layer (slim_yolo_v2.py:61) */
    /* ABI 2: the four fields below are all 0 for slim_yolo_v2 (a plain chain of 3x3 convolutions).  They describe what
     * yolo_v2 / darknet19 adds (models/yolo_v2.py:29-40,165-177, backbone/darknet.py:40-108, utils/modules.py:43-57): */
    int32_t ksize;        /* 0 or 3 = 3x3 pad 1; 1 = 1x1 (darknet19 bottlenecks, route_layer, yolo_v2's pred) */
    int32_t in_from;      /* 0 = input is the previous layer's output; k > 0 = the output of layer k-1 BEFORE its max-pool
                             (yolo_v2: route_layer reads C_5, the map maxpool_5 also consumes) */
    int32_t reorg;        /* 1 = space-to-depth (stride 2) of this layer's output: consumers see [h/2][w/2][4*cout], channel
                             (2*dy+dx)*cout + c  <-  pixel (2y+dy, 2x+dx), channel c  (reorg_layer, utils/modules.py:43-57) */
    int32_t concat_with;  /* k > 0: the input is torch.cat([output of layer k-1 (after its reorg), <in_from / previous>], dim=1)
                             (yolo_v2.py:171-174).  Both parts are brought to the smaller of their two activation exponents
                             (round-half-even right shift of the finer one) before they meet. */
} yolo_b200_layer;

/* Runtime tables: the reference hard-codes these in yolo_forward.c:32-37; here they are data. */
typedef struct yolo_b200_params {
    int32_t num_layers;                              /* 10 for slim_yolo_v2 (yolo_forward.c:1202-1262) */
    yolo_b200_layer layers[YOLO_B200_MAX_LAYERS];
    int32_t scale_w[YOLO_B200_MAX_LAYERS];           /* log2 weight scale per layer      (yolo_forward.c:32) */
    int32_t scale_b[YOLO_B200_MAX_LAYERS];           /* log2 bias scale per layer        (yolo_forward.c:33) */
    int32_t scale_a[YOLO_B200_MAX_LAYERS + 1];       /* log2 activation scale, [0]=input (yolo_forward.c:34) */
    int32_t retune[YOLO_B200_MAX_LAYERS];            /* accumulator scale (contract F)   (yolo_forward.c:35) */
    int32_t contract;                                /* YOLO_B200_CONTRACT_*  */
    int32_t round_mode;                              /* YOLO_B200_ROUND_* (contract F only) */
    int32_t head_mode;                               /* YOLO_B200_HEAD_*      */
    int32_t num_anchors;                             /* 5  (yolo_forward.c:36) */
    int32_t num_classes;                             /* 2  (slim_yolo_v2.py:87: 35 = 5*(1+4+2)) */
    int32_t stride;                                  /* 16 (yolo_forward.c:37, slim_yolo_v2.py:52) */
    float   anchors[YOLO_B200_MAX_ANCHORS][2];       /* (w,h) in grid cells (data/config.py:10-14) */
    float   conf_thresh;                             /* yolo_forward.c:1265 / test.py:22 */
    float   nms_thresh;                              /* yolo_forward.c:1265 / test.py:24 */
    int32_t max_det;                                 /* capacity of the per-frame detection list */
} yolo_b200_params;

/* One detection. HEAD_PYTHON: x1,y1,x2,y2 normalised to [0,1] (slim_yolo_v2.py:349).
 * HEAD_C: integer pixel corners stored as floats (struct BOX, yolo_forward.c:47-55). */
typedef struct yolo_b200_det {
    float x1, y1, x2, y2;
    float score;
    int32_t cls;
    int32_t anchor_index;   /* (row*W + col)*A + a: position in the reference's flat anchor order */
    int32_t pad_;
} yolo_b200_det;

typedef struct yolo_b200_ctx yolo_b200_ctx;

/* ---- library / context ---------------------------------------------------------------- */

/* Version of this ABI (bumped on incompatible change). */
int yolo_b200_abi_version(void);   /* 2 */

/* Thread-local text of the last error returned on this thread. */
const char *yolo_b200_last_error(void);

/* Channel stride used for a feature map of c logical channels: c rounded up to 16 (input: 4). */
int yolo_b200_cstride(int c);

/* Fill *p with the slim_yolo_v2 architecture and the tables exactly as shipped in
 * yolo_forward.c:32-37 (scale_a[0] = 0: the literal `65536` overflows `const char`),
 * COCO anchors, conf 0.01 / nms 0.5 (yolo_forward.c:1265), contract F, RNE, HEAD_PYTHON. */
int yolo_b200_default_params(yolo_b200_params *p);

/* Create a context on CUDA device `device` (one context per GPU; thread-compatible).
 * Fails (returns <0) when no sm_100 device is usable: there is no CPU fallback. */
int yolo_b200_create(yolo_b200_ctx **out, int device);
void yolo_b200_destroy(yolo_b200_ctx *ctx);

/* Use an existing CUDA stream (cudaStream_t cast to void*); NULL = the context's own (non-blocking) stream.
 * To run on the legacy default stream pass cudaStreamLegacy ((void*)0x1), not NULL. */
int yolo_b200_set_stream(yolo_b200_ctx *ctx, void *cuda_stream);

/* Replaces the `#include "weight.h"` data symbols w_conv0..9 / b_conv0..9 and the tables of
 * yolo_forward.c:5,32-37,1204-1260.  Host pointers; weights are repacked ONCE into the tile
 * layouts the kernels consume and copied to the device. */
int yolo_b200_load(yolo_b200_ctx *ctx, const int8_t *const *weights, const int8_t *const *biases,
                   const yolo_b200_params *params, int weight_layout);

/* Which convolution kernels run: 0 = auto (the weight-stationary tcgen05 kernel wherever the layer's packed weights fit
 * in shared memory, the streaming tcgen05 implicit GEMM for the other tensor-core shapes, the warp-level integer-MMA
 * kernel for the 3-channel first layer), 1 = integer dot-product (dp4a) kernels everywhere, 2 = streaming tcgen05 kernel only
 * (error for layers without a tensor-core shape), 3 = as 2 with the integer epilogue forced (the fp32 exact-rounding
 * epilogue is the default where the exponents allow it), 4 = weight-stationary tcgen05 kernel only, 5 = as 4 with the
 * integer epilogue forced.  All are CUDA; results are identical. */
int yolo_b200_set_conv_backend(yolo_b200_ctx *ctx, int backend);

/* Host-buffer entry points (yolo_b200_forward_rgb444 / _int8 / _f32 / _u8bgr) split a batch into chunks of `frames` frames
 * and overlap the host-to-device copy of chunk k+1 with the convolution layers of chunk k; decode + NMS run once over the
 * whole batch.  Default 64; 0 = one chunk (no overlap).  Results do not depend on it (frames are independent). */
int yolo_b200_set_host_chunk(yolo_b200_ctx *ctx, int frames);

/* Change thresholds / head mode after load (test.py --conf_thresh / --nms_thresh). */
int yolo_b200_set_thresholds(yolo_b200_ctx *ctx, float conf_thresh, float nms_thresh);

/* ---- whole-frame forward, HOST buffers (copies are part of the call) -------------------- */

/* Replaces yolo_forward() body, yolo_forward.c:1181-1279, for n frames of h x w RGB444.
 * dets: [n][max_det], counts: [n].  Only the filled part of each list is copied back: entries of frame i at index
 * >= counts[i] are unspecified (all host-buffer entry points). */
int yolo_b200_forward_rgb444(yolo_b200_ctx *ctx, const uint16_t *frames, int n, int h, int w,
                             yolo_b200_det *dets, int32_t *counts);

/* Asynchronous pair for a stream of batches (the camera loop of main.c:44-49 calls yolo_forward once per frame buffer while
 * the other buffer fills; here the unit is a batch).  yolo_b200_submit_* queues the whole call (copies, layers, decode + NMS)
 * and returns a ticket >= 0 without waiting; yolo_b200_wait(ticket) returns once dets / counts of that call are filled.
 * Up to two calls may be in flight: the tail of call i (the last chunk's layers, decode + NMS, the copy of the detections)
 * then overlaps the host-to-device copy of call i + 1, which keeps the PCIe link busy across calls.  `frames`, `dets` and
 * `counts` belong to the library between submit and wait (pinned host memory is needed for the copies to be asynchronous).
 * Results are those of the blocking call.  Errors: negative status; E_STATE (-2) when two calls are already in flight. */
int yolo_b200_submit_rgb444(yolo_b200_ctx *ctx, const uint16_t *frames, int n, int h, int w,
                            yolo_b200_det *dets, int32_t *counts);
int yolo_b200_submit_u8bgr(yolo_b200_ctx *ctx, const uint8_t *bgr, int n, int h, int w,
                           yolo_b200_det *dets, int32_t *counts);
int yolo_b200_wait(yolo_b200_ctx *ctx, int ticket);

/* Same from already-quantised int8 NHWC4 input (what camera_to_inpBuf writes, yolo_forward.c:87-123). */
int yolo_b200_forward_int8(yolo_b200_ctx *ctx, const int8_t *nhwc4, int n, int h, int w,
                           yolo_b200_det *dets, int32_t *counts);

/* Replaces the image front end of the Python path for images already at network size: BaseTransform without the resize
 * (data/__init__.py:30-56: /255, -mean, /std on the BGR bytes cv2 delivers), the BGR->RGB / CHW swap of test.py:79 and
 * a_tracker_in's quantisation (slim_yolo_v2.py:218,35), then the forward pass.  bgr: uint8 [n][h][w][3].
 * The three steps are a pure function of one byte per channel and run as a table lookup fused into the first layer. */
int yolo_b200_forward_u8bgr(yolo_b200_ctx *ctx, const uint8_t *bgr, int n, int h, int w,
                            yolo_b200_det *dets, int32_t *counts);

/* The reference's whole image front end: base_transform's `cv2.resize(image, (size[1], size[0]))` (data/__init__.py:36,
 * default INTER_LINEAR, reached through BaseTransform.__call__ :55 from test.py:76 / demo.py:71) followed by everything
 * yolo_b200_forward_u8bgr does.  bgr: uint8 [n][sh][sw][3] host images of one size (what cv2.imread / a capture loop
 * delivers); they are copied to the GPU as they are, resized there to the network size h x w chunk by chunk (between the
 * copy and the first layer) and never visit the host again.  The resize is bit-exact with OpenCV's 8-bit bilinear
 * (11-bit fixed-point taps; exact 2x decimation = 2x2 mean as OpenCV does).  sh == h && sw == w: no resize. */
int yolo_b200_forward_u8bgr_resize(yolo_b200_ctx *ctx, const uint8_t *bgr, int n, int sh, int sw, int h, int w,
                                   yolo_b200_det *dets, int32_t *counts);

/* The same for a batch of images of DIFFERENT sizes (a folder of image files, the VOC evaluator): one call, the chunked
 * copies, one batch-wide decode + NMS, as for one size.  src_hw: HOST int32 [n][2] = (sh, sw) of each image; the images are
 * packed back to back, image i at byte offset 3 * sum_{j<i} sh_j * sw_j, no padding, no alignment requirement.  Each image is
 * resized to h x w (bit-exact as above); boxes are normalised, so image i scales them by its own [sw, sh, sw, sh].
 * Errors: n < 0, sh or sw < 1, src_hw NULL with n > 0, null buffers: E_ARG (-1); an image over 2 GiB: E_UNSUPPORTED (-3).
 * n == 0 writes nothing.  The submit form is the asynchronous pair of yolo_b200_submit_u8bgr (needs n >= 1; + yolo_b200_wait). */
int yolo_b200_forward_u8bgr_ragged(yolo_b200_ctx *ctx, const uint8_t *bgr, int n, const int32_t *src_hw, int h, int w,
                                   yolo_b200_det *dets, int32_t *counts);
int yolo_b200_submit_u8bgr_ragged(yolo_b200_ctx *ctx, const uint8_t *bgr, int n, const int32_t *src_hw, int h, int w,
                                  yolo_b200_det *dets, int32_t *counts);

/* Camera and video frames in YUV, as decoders and webcams deliver them: each frame is converted to BGR exactly as
 * cv2.cvtColor(frame, COLOR_YUV2BGR_NV12 / _I420 / _YUYV) does (BT.601 limited range) and resized exactly as
 * yolo_b200_forward_u8bgr_resize does, on the GPU, in one pass, chunk by chunk between the copy and the first layer; the
 * rest is yolo_b200_forward_u8bgr_resize, so the results equal it run on the cvtColor'd frames.  4:2:0 frames cross the
 * host-to-device link at 1.5 bytes per pixel and YUYV at 2, against 3 for BGR.  Frames use cv2's Mat layout and are packed
 * at yolo_b200_yuv_frame_bytes() with no padding (frame i at byte i * frame_bytes):
 *   NV12: Y plane sh x sw, then sh/2 rows of sw bytes U,V interleaved           sh, sw even
 *   I420: Y plane, then the U plane (sh/2) x (sw/2), then the V plane            sh, sw even
 *   YUYV: sh rows of 2*sw bytes, macropixel Y0 U Y1 V                            sw even
 * sh == h && sw == w converts without resizing.  Errors: unknown format, odd sizes where the format needs even ones,
 * n < 0, sh / sw / h / w < 1, null buffers: E_ARG (-1); a frame over 2 GiB: E_UNSUPPORTED (-3).  n == 0 writes nothing.
 * The submit form is the asynchronous pair of yolo_b200_submit_u8bgr (needs n >= 1; + yolo_b200_wait). */
#define YOLO_B200_YUV_NV12  0
#define YOLO_B200_YUV_I420  1
#define YOLO_B200_YUV_YUYV  2
/* Bytes of one frame of this format and size (host only, no GPU needed), or a negative error as above. */
int yolo_b200_yuv_frame_bytes(int format, int sh, int sw);
int yolo_b200_forward_yuv(yolo_b200_ctx *ctx, const uint8_t *frames, int format, int n, int sh, int sw, int h, int w,
                          yolo_b200_det *dets, int32_t *counts);
int yolo_b200_submit_yuv(yolo_b200_ctx *ctx, const uint8_t *frames, int format, int n, int sh, int sw, int h, int w,
                         yolo_b200_det *dets, int32_t *counts);

/* Raw sensor frames in a Bayer mosaic, 8 bits per pixel, as machine-vision and embedded camera modules deliver them: each
 * frame is demosaiced to BGR exactly as cv2.cvtColor(frame, code) does with OpenCV's default bilinear demosaic, and
 * resized exactly as yolo_b200_forward_u8bgr_resize does, on the GPU, in one pass, chunk by chunk between the copy and the
 * first layer; the rest is yolo_b200_forward_u8bgr_resize, so the results equal it run on the cvtColor'd frames.  A frame
 * crosses the host-to-device link at 1 byte per pixel, against 3 for BGR.  Frames are uint8 [n][sh][sw], frame i at byte
 * i * sh * sw, no padding, no alignment requirement.  The pattern is named by the sensor's top-left 2x2 (GenICam and
 * ffmpeg name it so; OpenCV's legacy names count from the second row and column):
 *   RGGB: cv2 COLOR_BayerRGGB2BGR = COLOR_BayerBG2BGR, ffmpeg bayer_rggb8, GenICam BayerRG8
 *   BGGR: cv2 COLOR_BayerBGGR2BGR = COLOR_BayerRG2BGR, ffmpeg bayer_bggr8, GenICam BayerBG8
 *   GRBG: cv2 COLOR_BayerGRBG2BGR = COLOR_BayerGB2BGR, ffmpeg bayer_grbg8, GenICam BayerGR8
 *   GBRG: cv2 COLOR_BayerGBRG2BGR = COLOR_BayerGR2BGR, ffmpeg bayer_gbrg8, GenICam BayerGB8
 * sh == h && sw == w demosaics without resizing.  Errors: unknown pattern, n < 0, sh or sw < 3, h or w < 1, null buffers:
 * E_ARG (-1); a frame over 2 GiB: E_UNSUPPORTED (-3).  n == 0 writes nothing.  The submit form is the asynchronous pair of
 * yolo_b200_submit_u8bgr (needs n >= 1; + yolo_b200_wait). */
#define YOLO_B200_BAYER_RGGB  0
#define YOLO_B200_BAYER_BGGR  1
#define YOLO_B200_BAYER_GRBG  2
#define YOLO_B200_BAYER_GBRG  3
int yolo_b200_forward_bayer(yolo_b200_ctx *ctx, const uint8_t *frames, int pattern, int n, int sh, int sw, int h, int w,
                            yolo_b200_det *dets, int32_t *counts);
int yolo_b200_submit_bayer(yolo_b200_ctx *ctx, const uint8_t *frames, int pattern, int n, int sh, int sw, int h, int w,
                           yolo_b200_det *dets, int32_t *counts);

/* Frames in the pixel formats most other code holds: packed RGB (PIL, PyAV rgb24, dataset loaders), RGBA / BGRA (screen
 * capture, GUI toolkits, browsers, WebRTC, Android), 8-bit gray (monochrome machine-vision cameras, GenICam Mono8, thermal
 * cameras) and planar RGB (torch CHW uint8, torchvision.io.decode_image / decode_jpeg).  Each frame is converted to BGR
 * exactly as cv2.cvtColor does and resized exactly as yolo_b200_forward_u8bgr_resize does, on the GPU, in one pass, chunk
 * by chunk between the copy and the first layer; the rest is yolo_b200_forward_u8bgr_resize, so the results equal it run on
 * the cvtColor'd frames.  A gray frame crosses the host-to-device link at 1 byte per pixel and RGBA / BGRA at 4, against 3
 * for BGR.  Frames are packed at yolo_b200_pix_frame_bytes() with no padding (frame i at byte i * frame_bytes), no
 * alignment requirement (4-byte-aligned RGBA / BGRA sources take word loads, same results):
 *   RGB:        uint8 [sh][sw][3] R,G,B        cv2 COLOR_RGB2BGR,  ffmpeg rgb24
 *   RGBA:       uint8 [sh][sw][4] R,G,B,A      cv2 COLOR_RGBA2BGR, ffmpeg rgba    (alpha ignored)
 *   BGRA:       uint8 [sh][sw][4] B,G,R,A      cv2 COLOR_BGRA2BGR, ffmpeg bgra    (alpha ignored)
 *   GRAY:       uint8 [sh][sw]                 cv2 COLOR_GRAY2BGR, ffmpeg gray
 *   RGB_PLANAR: uint8 [3][sh][sw], planes R,G,B (torch CHW): cv2 COLOR_RGB2BGR of the HWC transpose; no ffmpeg name
 *               (ffmpeg's gbrp orders the planes G,B,R)
 * sh == h && sw == w converts without resizing.  Errors: unknown format, n < 0, sh / sw / h / w < 1, null buffers: E_ARG (-1);
 * a frame over 2 GiB: E_UNSUPPORTED (-3).  n == 0 writes nothing.  The submit form is the asynchronous pair of
 * yolo_b200_submit_u8bgr (needs n >= 1; + yolo_b200_wait). */
#define YOLO_B200_PIX_RGB        0
#define YOLO_B200_PIX_RGBA       1
#define YOLO_B200_PIX_BGRA       2
#define YOLO_B200_PIX_GRAY       3
#define YOLO_B200_PIX_RGB_PLANAR 4
/* Bytes of one frame of this format and size (host only, no GPU needed), or a negative error as above. */
int yolo_b200_pix_frame_bytes(int format, int sh, int sw);
int yolo_b200_forward_pix(yolo_b200_ctx *ctx, const uint8_t *frames, int format, int n, int sh, int sw, int h, int w,
                          yolo_b200_det *dets, int32_t *counts);
int yolo_b200_submit_pix(yolo_b200_ctx *ctx, const uint8_t *frames, int format, int n, int sh, int sw, int h, int w,
                         yolo_b200_det *dets, int32_t *counts);

/* Frames as decoders, cameras and array libraries lay them out: any of the formats above, one format and one size per
 * call, at a row pitch, plane offsets and a frame stride of the caller's choosing (NVDEC / PyNvVideoCodec / DALI surfaces,
 * cv2.cuda.GpuMat, V4L2 and GenICam buffers, FFmpeg AVFrame, strided numpy / torch views, and regions of a larger image).
 * Row r of plane p of frame i is at frames + i * frame_stride + plane_offset[p] + r * row_pitch[p].  The format decides the
 * planes and the bytes each row holds:
 *   BGR, RGB: 1 plane, sh rows of 3*sw     RGBA, BGRA: 1 plane, sh rows of 4*sw     gray, Bayer: 1 plane, sh rows of sw
 *   YUYV: 1 plane, sh rows of 2*sw          NV12: Y sh rows of sw, interleaved UV sh/2 rows of sw
 *   I420: Y sh rows of sw, U and V sh/2 rows of sw/2 each                        planar RGB: R, G, B, sh rows of sw each
 * Entries for planes the format lacks are ignored.  The results equal the family's packed call on the same frames compacted
 * (yolo_b200_forward_u8bgr_resize and the _yuv, _bayer and _pix entry points), byte for byte; packed frames are the layout
 * yolo_b200_frames_packed fills in.  Errors (E_ARG, -1): unknown family or format, sizes the format refuses, a negative stride or offset, a pitch
 * below the bytes of a row, n < 0, null pointers; E_UNSUPPORTED (-3): a frame spanning more than 2 GiB.  Frames may
 * overlap (frame_stride = 0 repeats one frame): the source is only read.
 * What a call reads: [frames + first, frames + end) of yolo_b200_frames_span, which the caller keeps addressable; nothing
 * outside it is read.  Inside it, the 3-byte and RGBA / BGRA word loads may touch padding between rows, but never use
 * it (weight 0).  RGBA / BGRA take word loads when every
 * row starts 4-byte aligned (frames + plane_offset[0], the pitch and the stride multiples of 4), bytes otherwise (same
 * results).  The host calls copy each chunk's span to the GPU as one copy, padding included: a generously padded layout
 * costs link time. */
#define YOLO_B200_SRC_BGR    0   /* format ignored: uint8 B,G,R pixels */
#define YOLO_B200_SRC_YUV    1   /* format = YOLO_B200_YUV_* */
#define YOLO_B200_SRC_BAYER  2   /* format = YOLO_B200_BAYER_* */
#define YOLO_B200_SRC_PIX    3   /* format = YOLO_B200_PIX_* */
typedef struct yolo_b200_frames {
    int32_t family, format;     /* YOLO_B200_SRC_*, the family's code */
    int32_t sh, sw;             /* source size in pixels */
    int64_t frame_stride;       /* bytes from frame i to frame i + 1 (>= 0) */
    int64_t plane_offset[3];    /* bytes from a frame's start to row 0 of plane p */
    int64_t row_pitch[3];       /* bytes from row r to row r + 1 of plane p */
} yolo_b200_frames;
/* Host only (no GPU needed): *d = the packed layout the family's entry points assume (frame i at i * frame bytes, planes
 * back to back, rows unpadded). */
int yolo_b200_frames_packed(yolo_b200_frames *d, int family, int format, int sh, int sw);
/* Host only: the bytes [frames + *first, frames + *end) a call over n frames of layout *d may read (n == 0: 0, 0). */
int yolo_b200_frames_span(const yolo_b200_frames *d, int n, int64_t *first, int64_t *end);
/* yolo_b200_forward_u8bgr_resize / _yuv / _bayer / _pix, and their submit form (+ yolo_b200_wait), on frames laid out as
 * *d says. */
int yolo_b200_forward_frames(yolo_b200_ctx *ctx, const uint8_t *frames, const yolo_b200_frames *d, int n, int h, int w,
                             yolo_b200_det *dets, int32_t *counts);
int yolo_b200_submit_frames(yolo_b200_ctx *ctx, const uint8_t *frames, const yolo_b200_frames *d, int n, int h, int w,
                            yolo_b200_det *dets, int32_t *counts);

/* Replaces SlimYOLOv2_quantize_bnfuse.forward(x, quantization=True) inference branch,
 * slim_yolo_v2.py:212-358, for a float NCHW batch (input quantised by a_tracker_in, :218). */
int yolo_b200_forward_f32(yolo_b200_ctx *ctx, const float *nchw, int n, int h, int w,
                          yolo_b200_det *dets, int32_t *counts);

/* ---- whole-frame forward, DEVICE buffers, asynchronous on the context stream ------------ */

int yolo_b200_forward_rgb444_dev(yolo_b200_ctx *ctx, const uint16_t *d_frames, int n, int h, int w,
                                 yolo_b200_det *d_dets, int32_t *d_counts);
int yolo_b200_forward_int8_dev(yolo_b200_ctx *ctx, const int8_t *d_nhwc4, int n, int h, int w,
                               yolo_b200_det *d_dets, int32_t *d_counts);
int yolo_b200_forward_f32_dev(yolo_b200_ctx *ctx, const float *d_nchw, int n, int h, int w,
                              yolo_b200_det *d_dets, int32_t *d_counts);
int yolo_b200_forward_u8bgr_dev(yolo_b200_ctx *ctx, const uint8_t *d_bgr, int n, int h, int w,
                                yolo_b200_det *d_dets, int32_t *d_counts);
int yolo_b200_forward_u8bgr_resize_dev(yolo_b200_ctx *ctx, const uint8_t *d_bgr, int n, int sh, int sw, int h, int w,
                                       yolo_b200_det *d_dets, int32_t *d_counts);
/* Images of different sizes packed back to back in device memory (layout and errors as yolo_b200_forward_u8bgr_ragged;
 * src_hw stays a HOST array).  Calls may be queued back to back without a synchronise: each call's resize tables are
 * written in stream order on the context stream. */
int yolo_b200_forward_u8bgr_ragged_dev(yolo_b200_ctx *ctx, const uint8_t *d_bgr, int n, const int32_t *src_hw, int h, int w,
                                       yolo_b200_det *d_dets, int32_t *d_counts);
/* YUV frames in device memory (layout and errors as yolo_b200_forward_yuv). */
int yolo_b200_forward_yuv_dev(yolo_b200_ctx *ctx, const uint8_t *d_frames, int format, int n, int sh, int sw, int h, int w,
                              yolo_b200_det *d_dets, int32_t *d_counts);
/* Bayer frames in device memory (layout and errors as yolo_b200_forward_bayer). */
int yolo_b200_forward_bayer_dev(yolo_b200_ctx *ctx, const uint8_t *d_frames, int pattern, int n, int sh, int sw, int h, int w,
                                yolo_b200_det *d_dets, int32_t *d_counts);

/* Frames of a pixel format in device memory (layout and errors as yolo_b200_forward_pix), e.g. torchvision's decoded
 * uint8 [3][sh][sw] tensors as YOLO_B200_PIX_RGB_PLANAR. */
int yolo_b200_forward_pix_dev(yolo_b200_ctx *ctx, const uint8_t *d_frames, int format, int n, int sh, int sw, int h, int w,
                              yolo_b200_det *d_dets, int32_t *d_counts);

/* Frames at a pitched layout in device memory (layout and errors as yolo_b200_forward_frames): a decoder surface, a
 * GpuMat or a strided CUDA tensor without a compacting copy. */
int yolo_b200_forward_frames_dev(yolo_b200_ctx *ctx, const uint8_t *d_frames, const yolo_b200_frames *d, int n, int h, int w,
                                 yolo_b200_det *d_dets, int32_t *d_counts);

/* Block until everything queued on the context stream is done. */
int yolo_b200_sync(yolo_b200_ctx *ctx);

/* ---- per-stage entry points (device buffers) -------------------------------------------- */

/* Input quantisers: pixel_norm_quantize (yolo_forward.c:57-85) as a 4096-entry table, and
 * a_tracker_in.quantize_activation (slim_yolo_v2.py:35: round-half-even of x*2^scale_a[0]).
 * Alignment of device buffers: int8 maps 16 bytes, fp32 input 16 bytes (error otherwise); camera frames 2 bytes
 * (frames that are not 16-byte aligned, or whose width is not a multiple of 4, take slower kernels, same results). */
int yolo_b200_quantize_rgb444(yolo_b200_ctx *ctx, const uint16_t *d_frames, int n, int h, int w,
                              int8_t *d_nhwc4);
int yolo_b200_quantize_f32(yolo_b200_ctx *ctx, const float *d_nchw, int n, int h, int w,
                           int8_t *d_nhwc4);
/* uint8 BGR image -> int8 NHWC4 (the front end of yolo_b200_forward_u8bgr as a stage), and its table for tests:
 * lut[ch*256 + v], ch 0..2 = R,G,B of the network input (R comes from BGR byte 2). */
int yolo_b200_quantize_u8bgr(yolo_b200_ctx *ctx, const uint8_t *d_bgr, int n, int h, int w, int8_t *d_nhwc4);
int yolo_b200_u8bgr_lut(yolo_b200_ctx *ctx, int8_t *lut_host);
/* cv2.resize(image, (dw, dh)) of base_transform (data/__init__.py:36) as a stage: uint8 [n][sh][sw][3] ->
 * uint8 [n][dh][dw][3], device buffers, any channel order (the three bytes are treated alike).  Needs no loaded network.
 * d_dst 4-byte aligned and dw a multiple of 4 take the vectorised kernel (same results otherwise). */
int yolo_b200_resize_u8bgr(yolo_b200_ctx *ctx, const uint8_t *d_src, int n, int sh, int sw,
                           uint8_t *d_dst, int dh, int dw);
/* The same for images of different sizes packed back to back in d_src (src_hw: HOST int32 [n][2] = (sh, sw) of each image,
 * image i at byte offset 3 * sum_{j<i} sh_j * sw_j) -> uint8 [n][dh][dw][3]; one kernel launch whatever the number of sizes.
 * Errors as yolo_b200_forward_u8bgr_ragged; n == 0 writes nothing. */
int yolo_b200_resize_u8bgr_ragged(yolo_b200_ctx *ctx, const uint8_t *d_src, int n, const int32_t *src_hw,
                                  uint8_t *d_dst, int dh, int dw);
/* The front end of yolo_b200_forward_yuv as a stage: n YUV frames (layout as there) -> uint8 BGR [n][dh][dw][3], equal to
 * cv2.resize(cv2.cvtColor(frame, code), (dw, dh)); one kernel launch, nothing written at source resolution.  Needs no
 * loaded network; no alignment requirement (d_dst 4-byte aligned and dw a multiple of 4 take word stores). */
int yolo_b200_yuv_to_bgr_resize(yolo_b200_ctx *ctx, const uint8_t *d_src, int format, int n, int sh, int sw,
                                uint8_t *d_dst, int dh, int dw);
/* The front end of yolo_b200_forward_bayer as a stage: n Bayer frames (layout as there) -> uint8 BGR [n][dh][dw][3], equal
 * to cv2.resize(cv2.cvtColor(frame, code), (dw, dh)); one kernel launch, nothing written at source resolution.  Needs no
 * loaded network; no alignment requirement (d_dst 4-byte aligned and dw a multiple of 4 take word stores). */
int yolo_b200_bayer_to_bgr_resize(yolo_b200_ctx *ctx, const uint8_t *d_src, int pattern, int n, int sh, int sw,
                                  uint8_t *d_dst, int dh, int dw);
/* The front end of yolo_b200_forward_pix as a stage: n frames of a pixel format (layout as there) -> uint8 BGR
 * [n][dh][dw][3], equal to cv2.resize(cv2.cvtColor(frame, code), (dw, dh)); one kernel launch, nothing written at source
 * resolution.  Needs no loaded network; no alignment requirement (d_dst 4-byte aligned and dw a multiple of 4 take word
 * stores). */
int yolo_b200_pix_to_bgr_resize(yolo_b200_ctx *ctx, const uint8_t *d_src, int format, int n, int sh, int sw,
                                uint8_t *d_dst, int dh, int dw);
/* The front end of yolo_b200_forward_frames as a stage: n frames laid out as *d says (device memory) -> uint8 BGR
 * [n][dh][dw][3], equal to the family's stage on the frames compacted; one kernel launch.  Needs no loaded network. */
int yolo_b200_frames_to_bgr_resize(yolo_b200_ctx *ctx, const uint8_t *d_src, const yolo_b200_frames *d, int n,
                                   uint8_t *d_dst, int dh, int dw);
/* Host only (no GPU needed), for tests: the per-index programme of that resize along one axis, taps[4*d + {0,1,2,3}] =
 * (source index 0, source index 1, weight 0, weight 1), weights in units of 1/2048; horizontal != 0 re-anchors the tap
 * at the image border as OpenCV's horizontal pass does. */
int yolo_b200_resize_taps(int src, int dst, int horizontal, int32_t *taps);
/* The 4096 x 4 byte table itself (host copy), for tests: lut[code*4 + {0,1,2}] = R,G,B. */
int yolo_b200_rgb444_lut(yolo_b200_ctx *ctx, int8_t *lut_host);

/* One layer: replaces first_conv / second_conv / conv_normal / conv_last
 * (yolo_forward.c:269,420,575,772) and Conv2d_fuse + tracker + pool (slim_yolo_v2.py:220-328).
 * d_in is [n][h][w][cstride(cin)] (layer 0: [n][h][w][4]); d_out is [n][h'][w'][cstride(cout)]. */
int yolo_b200_conv_layer(yolo_b200_ctx *ctx, int layer, const int8_t *d_in, int n, int h, int w,
                         int8_t *d_out);

/* Test hook: apply layer l's epilogue arithmetic (bias add, shifts, saturation, leaky-ReLU; no pool) to `count`
 * caller-supplied int32 accumulators; element i uses the bias of channel i % cout.  Returns which implementation
 * ran: 0 = integer, 1 = exact-fp32 contract F, 2 = exact-fp32 contract P, 3 = as 1 without the (provably redundant)
 * upper 16-bit clamp (or < 0 on error). */
int yolo_b200_debug_requant(yolo_b200_ctx *ctx, int layer, const int32_t *d_acc, size_t count, int8_t *d_out,
                            int force_generic);

/* All layers; returns the device pointer of the last layer's output (owned by the context,
 * valid until the next call) and its grid size. */
int yolo_b200_backbone(yolo_b200_ctx *ctx, const int8_t *d_nhwc4, int n, int h, int w,
                       const int8_t **d_pred, int *gh, int *gw);
/* Calibration on the GPU: one forward pass over a float NCHW calibration batch with fresh trackers.  Replaces the
 * calibration call of retune_bias_quantize.py -q (AveragedRangeTracker first-call rule, slim_yolo_v2.py:22-27,33:
 * scale_a = floor(log2(127 / max|a|)) per activation) and the overflow search of retune_bias_quantize_findbest.py
 * (retune[l] = largest r with max|y_l| * 2^r < 2^15, slim_yolo_v2.py:222-227).  Updates the context's tables and epilogue
 * programmes in place and returns them (scale_a_out: num_layers + 1 entries, retune_out: num_layers; either may be NULL). */
int yolo_b200_calibrate_f32(yolo_b200_ctx *ctx, const float *d_nchw, int n, int h, int w,
                            int32_t *scale_a_out, int32_t *retune_out);

/* Several calibration batches (trainable / un-frozen trackers, slim_yolo_v2.py:28-31): every tracker that has been called
 * before (tracker_scale[t] != 0) moves by the exponential average scale <- scale * (1 - momentum) + (127 / max|a|) * momentum
 * in float32 as the reference's tensor ops do, the others take the first-call rule; the exponent in force becomes
 * floor(log2(scale)) (:33).  tracker_scale: num_layers + 1 floats = the `scale` buffers of a_tracker_in .. a_tracker_pred, in
 * and out (all zero = fresh trackers = yolo_b200_calibrate_f32, which also fixes retune[]).  On any error the context keeps
 * the tables it had. */
int yolo_b200_update_trackers_f32(yolo_b200_ctx *ctx, const float *d_nchw, int n, int h, int w, float momentum,
                                  float *tracker_scale, int32_t *scale_a_out, int32_t *retune_out);

/* The `find=True` overflow probe (slim_yolo_v2.py:222-226, repeated for every layer up to :327;
 * retune_bias_quantize_findbest.py:364): one forward pass with the tables in force, nothing changes; max_abs[0] = max|x| of
 * the input, max_abs[l + 1] = max|y_l| of layer l's output after the leaky-ReLU and before its tracker (exact: the
 * activations are dyadic rationals).  num_layers + 1 doubles. */
int yolo_b200_measure_f32(yolo_b200_ctx *ctx, const float *d_nchw, int n, int h, int w, double *max_abs);

/* Copy layer l's output of the most recent backbone call to the host (debug / parity). */
int yolo_b200_get_layer_output(yolo_b200_ctx *ctx, int layer, int8_t *host_out, size_t bytes);

/* Head: replaces get_boxes + conf_sort + NMS (yolo_forward.c:1052-1147) and
 * decode_boxes + postprocess + nms (slim_yolo_v2.py:111-210,330-358).
 * d_pred: [n][gh][gw][cstride(A*(5+C))]. in_h/in_w: network input size (box normalisation). */
int yolo_b200_detect(yolo_b200_ctx *ctx, const int8_t *d_pred, int n, int gh, int gw,
                     int in_h, int in_w, yolo_b200_det *d_dets, int32_t *d_counts);

/* ---- multi-GPU collection of the detection lists (SURVEY 8e: frames are sharded, only the lists are gathered) -------------
 * The reference has no counterpart (one camera, one accelerator).  The lists travel to ONE collecting GPU over NVLink by
 * copy-engine peer writes: no collective kernel competes with the persistent convolution CTAs for SMs. */

/* Squeeze the fixed-capacity lists to their filled part: d_offsets[f] = records of the frames before f (d_offsets[n] = total,
 * n + 1 entries), d_packed[d_offsets[f] + i] = d_dets[f][i] for i < min(d_counts[f], max_det).  Asynchronous on the context stream. */
int yolo_b200_pack_detections(yolo_b200_ctx *ctx, const yolo_b200_det *d_dets, const int32_t *d_counts, int n,
                              yolo_b200_det *d_packed, int32_t *d_offsets);
/* A device buffer other processes of this node can write: cudaMalloc + cudaIpcGetMemHandle (64-byte handle to hand to the peers). */
int yolo_b200_ipc_alloc(yolo_b200_ctx *ctx, size_t bytes, void **d_ptr, unsigned char handle[64]);
/* Map a peer's buffer into this process (cudaIpcOpenMemHandle with lazy peer access). */
int yolo_b200_ipc_open(yolo_b200_ctx *ctx, const unsigned char handle[64], void **d_ptr);
/* Release: opened != 0 unmaps a peer's buffer, opened == 0 frees a buffer made by yolo_b200_ipc_alloc. */
int yolo_b200_ipc_close(yolo_b200_ctx *ctx, void *d_ptr, int opened);
/* cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault) on `cuda_stream` (NULL = the context stream): device, peer-device or
 * pinned-host memory on either side; between GPUs it runs on a copy engine. */
int yolo_b200_copy_async(yolo_b200_ctx *ctx, void *dst, const void *src, size_t bytes, void *cuda_stream);

/* Sticky count of int8 saturations in contract P (the reference never clamps,
 * slim_yolo_v2.py:35; non-zero means the result may differ from it). Resets on read. */
int yolo_b200_overflow_count(yolo_b200_ctx *ctx, int64_t *count);

/* Number of kernels this library launched on the context since creation (bench bookkeeping). */
int64_t yolo_b200_launch_count(yolo_b200_ctx *ctx);
/* How many of those launches, in the automatic back end, fell to the integer dot-product kernel because no tensor-core kernel
 * takes the layer's shape or the buffers' alignment (a first layer wider than 16 channels, a 2-byte-aligned frame pointer, a
 * map width that is not a multiple of 4 ...).  Same results, lower speed: 0 on the benchmarked configurations. */
int64_t yolo_b200_slow_path_count(yolo_b200_ctx *ctx);

/* Device time of the most recent yolo_b200_backbone()/forward call per layer, in ms
 * (CUDA events on the context stream; enabled by yolo_b200_enable_timing). */
int yolo_b200_enable_timing(yolo_b200_ctx *ctx, int enable);
int yolo_b200_layer_times_ms(yolo_b200_ctx *ctx, float *ms, int capacity);

/* ---- host-side helpers of the reference's tail -------------------------------------------- */

/* draw_rectangle (yolo_forward.c:1149-1178), restated WITHOUT its out-of-bounds index arithmetic:
 * draws 1-pixel box outlines into an RGB444 frame, red (0x000f) for class 0, green (0x00f0) otherwise. */
int yolo_b200_draw_rectangles(uint16_t *frame, int h, int w, const yolo_b200_det *dets, int count,
                              int boxes_are_normalised);

/* Legacy symbol, identical signature to yolo_forward.c:1181-1183, called from the camera ISR
 * (main.c:44-49) as yolo_forward(18,22,16,20,32,16, camera_bram, vga_bram).  The tile arguments
 * describe FPGA buffers and are validated (TRow==Tr+2, TCol==Tc+2) then ignored.  Uses the
 * process-wide default context installed by yolo_b200_set_default_context(); draws the detections
 * into the camera buffer and copies it to the VGA buffer (76800 pixels), as the reference does
 * (yolo_forward.c:1280-1281). */
void yolo_forward(const char TRow, const char TCol, const char Tr, const char Tc,
                  const char Tm, const char Tn,
                  short int *camera_bram_pointer, int *vga_bram_pointer);
int yolo_b200_set_default_context(yolo_b200_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* YOLO_B200_H */
