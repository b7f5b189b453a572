// kernels.h — internal launch interface between the host library (yolo_b200.cu) and the kernel files.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"
#include "../../include/yolo_b200.h"

namespace yb {

struct ConvArgs {
    const int8_t *in;      // [n][H][W][cs_in]
    int n, H, W, cs_in;
    const int8_t *wgt;     // [cout_pad][9][cs_in]  (cout_pad: multiple of 32, zero padded)
    const int8_t *wgt_k160; // cs_in == 16 only: [cout_pad][10][16], 10th tap all zero (two taps per K=32 MMA)
    const uint8_t *wgt_swz = nullptr;  // cs_in % 128 == 0: [9*cs_in/128][cs_out][128 B] blocks in the 128B-swizzled smem layout (conv_umma.cu)
    int wgt_swz_rows = 0;              // rows per block of wgt_swz (= cs_out)
    const uint8_t *wimg;   // cs_in >= 16: UMMA no-swizzle core-matrix image of the weights for conv_ws.cu (see pack_wimg)
    const uint8_t *wimg_tap;   // cs_in 128 / 256: the same image tap-major, [tap][128-channel plane][cs_out/8][8][8][16 B] (conv_ws.cu, weight streaming)
    const uint8_t *wimg_tap2 = nullptr; // cs_in 128 / 256, cs_out 256: [half of cs_out][plane][tap][128/8][8][8][16 B] chunks of 16 KB (conv_wsp.cu)
    const uint8_t *wimg_tap3 = nullptr; // 3x3, cs_in % 128 == 0, cs_out % 256 == 0, wider than 256: [slice of 256][half][plane][tap] chunks of 16 KB (conv_ws3.cu)
    const uint8_t *wimg_rp = nullptr;  // cs_in == 16, cs_out == 32, pooled: row-pair image [2*cs_out/8][12][8][16 B] (conv_rp.cu)
    const uint8_t *wimg_rps = nullptr; // the same for an x-split input map (chunk order (row, kw 0), (row, kw 2) x 4 rows, then (row, kw 1) x 4)
    int w_rows;            // cout_pad
    int bias_abs_max;      // max |bias_sh[c]| (decides whether the exact fp32 epilogue applies)
    int force_generic_epilogue;   // tests: run the integer epilogue even where the fp32 one applies
    const int *bias_sh;    // [cout_pad] pre-shifted bias (see LayerQ)
    int cout, cs_out;
    LayerQ q;
    int8_t *out;           // [n][H'][W'][cs_out]
    unsigned *ovf;         // contract-P saturation counter
    int *stats = nullptr;  // conv3x3_direct only: calibration pass, see conv_direct.cu (bias_sh then holds b << lb, q.la the shift)
    int out_xsplit = 0;    // conv_first.cu (pooled, 16 output channels, even output width): rows stored split by x parity, [even pixels][odd pixels]
    int in_xsplit = 0;     // conv_rp.cu: the input map is stored that way
    int taps = 9;          // conv_umma.cu only: 9 = 3x3, 1 = 1x1 (then wgt / wgt_swz hold ONE tap: [cout_pad][cs_in] / [cs_in/128][cs_out][128])
    const int8_t *wgt1 = nullptr;   // taps == 1: [cout_pad][cs_in]
};

// conv_direct.cu
cudaError_t conv3x3_direct(const ConvArgs &a, cudaStream_t st);

// The input kinds of the network: int8 NHWC4, RGB444 uint16 frames (+ 4096-word table), uint8 BGR images (+ 3x256-byte
// table), float NCHW.  The first three are also the first-layer kernels' source template argument; f32 is quantised first.
enum InKind { IN_INT8 = 0, IN_RGB444 = 1, IN_BGR = 2, IN_F32 = 3 };

// conv_first.cu (first layer: NHWC4 input, <= 16 output channels, warp-level integer MMAs)
bool conv3x3_first_supported(const ConvArgs &a);
bool conv3x3_first_src_ok(InKind src_kind, const void *src);    // pointer alignment the first-layer kernel needs
// src_kind IN_INT8 reads a.in; IN_RGB444 / IN_BGR read src with the context's table lut for that source
cudaError_t conv3x3_first(const ConvArgs &a, cudaStream_t st, InKind src_kind = IN_INT8, const void *src = nullptr, const void *lut = nullptr);

// conv_fs.cu (first layer on tcgen05: 3 -> 16 channels + pool for pooled widths >= 128; src_kind IN_INT8, IN_RGB444 or IN_BGR)
bool conv3x3_fs_supported(const ConvArgs &a, InKind src_kind, const void *src);
cudaError_t conv3x3_fs(const ConvArgs &a, cudaStream_t st, InKind src_kind, const void *src, const void *lut);

// conv_umma.cu (tcgen05 / TMEM / TMA implicit GEMM)
bool conv3x3_umma_supported(const ConvArgs &a);
cudaError_t conv3x3_umma(const ConvArgs &a, cudaStream_t st, int sm_count);
cudaError_t requant_probe(const ConvArgs &a, const int *acc, size_t count, int8_t *out, int *epi_used, cudaStream_t st);

// conv_ws.cu (weight-stationary tcgen05 kernel: weights resident in shared memory, haloed tile fetched once)
bool conv3x3_ws_supported(const ConvArgs &a);
cudaError_t conv3x3_ws(const ConvArgs &a, cudaStream_t st, int sm_count);

// conv_wsp.cu (pair-streamed tcgen05 kernel for the deep narrow layers: each streamed weight chunk feeds two 128-pixel tiles)
bool conv3x3_wsp_supported(const ConvArgs &a);
cudaError_t conv3x3_wsp(const ConvArgs &a, cudaStream_t st, int sm_count);

// conv_ws2.cu (CTA-pair tcgen05 kernel, cta_group::2: each SM of a pair holds one 128-pixel tile and half of the weights)
bool conv3x3_ws2_supported(const ConvArgs &a, int sm_count);
cudaError_t conv3x3_ws2(const ConvArgs &a, cudaStream_t st, int sm_count);

// conv_ws3.cu (the CTA-pair kernel for the wide 3x3 layers of yolo_v2: units of (tile pair, 256-channel slice), halo planes streamed)
bool conv3x3_ws3_supported(const ConvArgs &a, int sm_count);
cudaError_t conv3x3_ws3(const ConvArgs &a, cudaStream_t st, int sm_count);

// conv_rp.cu (row-pair tcgen05 kernel for the thin pooled layers: two output rows in the GEMM N dimension, dense TMA-fed halo)
bool conv3x3_rp_supported(const ConvArgs &a);
bool conv3x3_rp_split_supported(const ConvArgs &a);      // the variant that reads an x-split input map (a.in_xsplit is ignored by the test)
cudaError_t conv3x3_rp(const ConvArgs &a, cudaStream_t st, int sm_count);

// graph.cu (yolo_v2: stand-alone max-pool, reorg + concat with exponent alignment)
cudaError_t maxpool2x2(const int8_t *in, int n, int H, int W, int cs, int8_t *out, cudaStream_t st);
cudaError_t concat_reorg(const int8_t *A, int cs_a, int ca, int reorg, int sh_a, const int8_t *B, int cs_b, int cb, int sh_b,
                         int n, int h, int w, int cs_out, int8_t *out, cudaStream_t st);

// quantize.cu
cudaError_t quantize_rgb444(const uint16_t *frames, size_t npix, const int *lut_dev, int8_t *nhwc4, cudaStream_t st);
cudaError_t quantize_u8bgr(const uint8_t *bgr, size_t npix, const uint8_t *lut8_dev, int8_t *nhwc4, unsigned *ovf, cudaStream_t st);
cudaError_t absmax_f32(const float *x, size_t count, unsigned *out_bits, cudaStream_t st);   // max |x| as float bits (atomicMax)
cudaError_t quantize_f32(const float *nchw, int n, int h, int w, int sa, int8_t *nhwc4, unsigned *ovf, cudaStream_t st);

// resize.cu (uint8 HxWx3 bilinear resize = cv2.resize of the reference's BaseTransform, data/__init__.py:36)
void resize_axis_table(int src, int dst, bool clamp_weights, int index_scale, int4 *out);   // host: (tap0, tap1, weight0, weight1) per output index
// xtab: per column (byte offset of tap 0 in its row, weight0 | weight1 << 16), tap 1 = the next pixel; ytab: per row (row 0, row 1, weight0 << 16, weight1 << 16)
// taps and weights of one geometry (sh, sw) -> (dh, dw) in that layout: ytab [dh], xtab [dw] (host)
void resize_geometry_tables(int sh, int sw, int dh, int dw, int4 *ytab, int2 *xtab);
// Source formats: the YUV layouts (NV12, I420, YUYV in cv2's Mat layout), uint8 BGR, and the Bayer mosaics (uint8 [sh][sw],
// RS_BAYER_* - RS_BAYER_RGGB = column flip | row flip << 1 relative to RGGB).  Camera frames (YUV, Bayer) are packed at
// camera_frame_bytes.
enum { RS_YUV_NV12 = YOLO_B200_YUV_NV12, RS_YUV_I420 = YOLO_B200_YUV_I420, RS_YUV_YUYV = YOLO_B200_YUV_YUYV, RS_BGR = 3,
       RS_BAYER_RGGB = 4, RS_BAYER_GRBG = 5, RS_BAYER_GBRG = 6, RS_BAYER_BGGR = 7 };
size_t camera_frame_bytes(int format, int sh, int sw);     // 0 for BGR or an unknown format
// Images of different sizes packed back to back in one buffer: frame f starts at byte off of src, its rows are
// pitch = 3 * sw bytes apart, and its tables are ytab + geom * dh, xtab + geom * dw.
struct alignas(16) ResizeFrame { unsigned long long off; int pitch; int geom; };
// One launch: n frames of format fmt -> uint8 BGR [n][dh][dw][3], bit-exact with cv2.resize (of cv2.cvtColor for YUV and Bayer).
// frames_dev == nullptr: the frames are sh x sw at a uniform stride from src, with the tables ytab [dh], xtab [dw].
// Otherwise (RS_BGR only) frames_dev[f] describes frame f as above.  A BGR launch reads no byte at or past src + src_bytes.
cudaError_t resize_u8c3(const uint8_t *src, size_t src_bytes, int fmt, const ResizeFrame *frames_dev, int n, int sh, int sw,
                        uint8_t *dst, int dh, int dw, const int2 *xtab_dev, const int4 *ytab_dev, int sm_count, cudaStream_t st);

// head.cu
struct HeadArgs {
    const int8_t *pred;    // [n][gh][gw][cs]
    int n, gh, gw, cs;
    int A, C;              // anchors per cell, classes
    int sa_pred;           // exponent of the prediction map
    float anchors[YOLO_B200_MAX_ANCHORS][2];
    int stride, in_h, in_w;
    float conf_thresh, nms_thresh;
    int head_mode;
    int max_det;
    int fused_decode = 0;  // head_nms decodes the prediction map itself (head_nms_fuses_decode): scores / cls / boxes are not read
    // scratch [n][N]: best-class score, class, box
    float *scores; int *cls; float4 *boxes;
    yolo_b200_det *dets;   // [n][max_det]
    int32_t *counts;       // [n]
};
constexpr int HEAD_MAX_CAND = 4096;   // candidates per frame the NMS kernel can hold in shared memory
cudaError_t head_decode(const HeadArgs &a, cudaStream_t st);
bool head_nms_fuses_decode(const HeadArgs &a);   // the python head's grid NMS kernel decodes in place: no head_decode launch, no scratch traffic
cudaError_t head_nms(const HeadArgs &a, cudaStream_t st);
cudaError_t head_init(void);          // one-time function attributes (dynamic shared memory)
cudaError_t pack_detections(const yolo_b200_det *dets, const int32_t *counts, int n, int max_det, yolo_b200_det *packed, int32_t *offsets, cudaStream_t st);

}  // namespace yb
