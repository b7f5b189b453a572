// yolo_b200.cu — host side of the C-ABI declared in include/yolo_b200.h.
//
// Owns device memory, repacks weights once at load, derives each layer's epilogue programme from the exponent
// tables (set_quantize_scale, c_embedding/yolo_forward.c:233-257) and sequences the kernels on one CUDA stream.
// There is no CPU fallback: every entry point that computes needs a CUDA device.
#include "kernels.h"
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <map>
#include <mutex>
#include <vector>
#include <string>

using namespace yb;

static thread_local char g_err[512] = "";
static int fail(int code, const char *fmt, ...)
{
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof g_err, fmt, ap); va_end(ap);
    return code;
}
#define CU(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return fail(-5, "%s: %s (%s:%d)", #x, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)

enum { E_ARG = -1, E_STATE = -2, E_UNSUPPORTED = -3, E_NOMEM = -4, E_CUDA = -5 };

struct LayerDev {
    int cin, cout, cs_in, cs_out, cout_pad;
    int ksize = 3, in_from = 0, reorg = 0, concat_with = 0;     // yolo_v2 / darknet19 graph fields (include/yolo_b200.h, ABI 2)
    bool unfused_pool = false;     // the max-pool runs as its own kernel: a route reads the un-pooled map, or the layer is wider than 256 channels
    int8_t *w1 = nullptr;          // ksize == 1: [cout_pad][cs_in] (conv_umma.cu, one tap)
    int8_t *raw = nullptr; size_t raw_cap = 0;      // un-pooled output when the pool is not fused
    int8_t *cat = nullptr; size_t cat_cap = 0;      // concatenated (+ reorganised, exponent-aligned) input of a concat layer
    int rh = 0, rw = 0;            // un-pooled output map of the most recent call
    std::vector<int8_t> wp_host;   // [cout_pad][9][cs_in] as repacked at load (the swizzled image is built on first use)
    int bias_abs_max = 0;
    std::vector<int8_t> bias_host;   // int8 biases as loaded (the epilogue programme is re-derived when the tables change)
    LayerQ q;
    int8_t *w = nullptr;       // [cout_pad][9][cs_in]
    int8_t *w_k160 = nullptr;  // cs_in == 16: [cout_pad][10][16] with a zero 10th tap (conv_umma.cu)
    uint8_t *wimg = nullptr;   // cs_in >= 16: core-matrix image [cs_out/8][kc][8][16] (conv_ws.cu)
    uint8_t *wimg_tap = nullptr;   // cs_in 128 / 256: chunk-major image [tap][plane][cs_out/8][8][8][16] (conv_ws.cu, streamed weights)
    uint8_t *wimg_tap2 = nullptr;  // cs_in 128 / 256, cs_out 256: 16 KB chunks [half][plane][tap] (conv_wsp.cu)
    uint8_t *wimg_tap3 = nullptr;  // wide 3x3 layers (yolo_v2): 16 KB chunks [slice][half][plane][tap] (conv_ws3.cu)
    uint8_t *wimg_rp = nullptr;    // cs_in == 16, cs_out == 32, pooled: row-pair image (conv_rp.cu)
    uint8_t *wimg_rps = nullptr;   // the same in the chunk order of the x-split variant
    bool xsplit = false;           // the most recent output map is stored with its rows split by x parity ([even pixels][odd pixels])
    uint8_t *w_swz = nullptr;  // cs_in % 128 == 0: 128B-swizzled blocks [9*cs_in/128][cs_out][128] (conv_umma.cu B operand)
    int *bias_sh = nullptr;    // [cout_pad]
    int8_t *out = nullptr;     // [n][h'][w'][cs_out] of the most recent backbone call
    int8_t *view = nullptr;    // where the most recent output actually lives (out, or a slot of the batch-wide prediction map)
    size_t out_cap = 0;
    int oh = 0, ow = 0;
};

// YOLO_B200_TRACE_HOST=1: timeline of one host-buffer call (ms since its start), printed to stderr
struct HostTrace {
    bool on = false;
    cudaEvent_t t0 = nullptr;
    std::vector<std::pair<std::string, cudaEvent_t>> ev;
    void mark(const char *what, int k, cudaStream_t st) {
        if (!on) return;
        cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st);
        ev.push_back({std::string(what) + " " + std::to_string(k), e});
    }
    void dump() {
        if (!on) return;
        for (auto &p : ev) { float ms = 0; cudaEventSynchronize(p.second); cudaEventElapsedTime(&ms, t0, p.second); fprintf(stderr, "  %-22s %7.3f ms\n", p.first.c_str(), ms); cudaEventDestroy(p.second); }
        cudaEventDestroy(t0);
    }
};

// Device tables of the resize front end (resize_tables): a table image uploaded in stream order through two alternating
// pinned staging buffers, so an upload waits for no queued resize and overwrites nothing a queued resize still reads.
struct ResizeTables {
    void *dev = nullptr; size_t dev_cap = 0;
    char *host[2] = {nullptr, nullptr}; size_t host_cap[2] = {0, 0};
    cudaEvent_t ev[2] = {nullptr, nullptr};                 // recorded after the copy out of host[k]
    int next = 0;
    long long key[10] = {};                                 // the context's uniform cache: (sh, sw, dh, dw) and the layout of its tables
    const ResizeFrame *frames = nullptr; const int4 *ytab = nullptr; const int2 *xtab = nullptr;     // inside dev
};

// One host-buffer call in flight: its device staging, batch-wide prediction map, detection lists, the pinned landing
// area of the counts and its events.  Two slots let the tail of call i (last chunk's layers, decode + NMS, copy of the
// detections) overlap the host-to-device copy of call i + 1 (yolo_b200_submit_* / yolo_b200_wait).
constexpr int YB_HOST_SLOTS = 2;
struct HostSlot {
    void *stage_in = nullptr; size_t stage_in_cap = 0;      // device staging of the host frames (network-size frames)
    void *rs_src = nullptr; size_t rs_src_cap = 0;          // resize front end: staged source images
    ResizeTables tabs;                                      // images of different sizes: descriptors + tables of the call (s_in)
    int8_t *pred_all = nullptr; size_t pred_all_cap = 0;    // batch-wide prediction map
    yolo_b200_det *d_dets = nullptr; size_t dets_cap = 0;
    int32_t *d_counts = nullptr; size_t counts_cap = 0;
    int32_t *counts_pinned = nullptr; size_t counts_pinned_cap = 0;   // counts land here first: the caller's array may be pageable
    std::vector<cudaEvent_t> ev_in, ev_done, ev_cnt;
    cudaEvent_t ev_out = nullptr;
    bool busy = false;
    // the call in flight
    int ngroups = 0, grp_f0[2] = {0, 0}, grp_n[2] = {0, 0};
    yolo_b200_det *dets = nullptr; int32_t *counts = nullptr;
    HostTrace tr;
};

struct yolo_b200_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    bool loaded = false;
    bool graph = false;                  // the network is not a plain chain of 3x3 convolutions (yolo_v2 / darknet19)
    int64_t slow_path_launches = 0;      // layers that fell back to the dot-product kernel in the auto back end
    yolo_b200_params prm;
    std::vector<LayerDev> layers;
    int *lut_dev = nullptr;              // 4096 packed (R,G,B,0) words
    int8_t lut_host[4096 * 4];
    uint8_t *lut8_dev = nullptr;         // uint8 BGR front end: [3][256] quantised bytes (R,G,B) + [3][256] saturation flags
    uint8_t lut8_host[1536];
    bool lut8_saturates = false;
    unsigned *ovf_dev = nullptr;
    int *stats_dev = nullptr;            // calibration: {max, min} of a layer's numerator / abs-max bits of the input
    int8_t *in_q = nullptr; size_t in_q_cap = 0;        // quantised NHWC4 input
    uint8_t *rs_out = nullptr; size_t rs_out_cap = 0;   // resize front end: resized images (device entry point)
    ResizeTables rs_cache;                              // one source size: the tables of the most recent geometry
    ResizeTables rs_call;                               // images of different sizes, device entry points: the most recent call's
    float *h_scores = nullptr; int *h_cls = nullptr; float4 *h_boxes = nullptr; size_t head_cap = 0;
    int last_n = 0;
    int64_t launches = 0;
    int sm_count = 148;
    int conv_backend = 0;                // 0 auto (tensor cores where the shape allows), 1 dp4a direct, 2 tcgen05 only
    bool timing = false;
    std::vector<cudaEvent_t> ev;
    int ev_used = 0;
    // host-buffer entry points: copies of chunk k+1 / k-1 overlap the kernels of chunk k
    cudaStream_t s_in = nullptr, s_out = nullptr, s_head = nullptr;
    int host_chunk = 64;                 // frames per chunk (measured best at 416x416: tools/t_e2e.py)
    HostSlot slots[YB_HOST_SLOTS];       // buffers of the host-buffer calls in flight (yolo_b200_submit_* / yolo_b200_wait)
};

static std::mutex g_default_mu;
static yolo_b200_ctx *g_default_ctx = nullptr;

#pragma GCC visibility push(default)     // only the C-ABI is exported from the shared library
extern "C" {

int yolo_b200_abi_version(void) { return 2; }
const char *yolo_b200_last_error(void) { return g_err; }
int yolo_b200_cstride(int c) { return c <= 4 ? 4 : (c + 15) / 16 * 16; }

int yolo_b200_default_params(yolo_b200_params *p)
{
    if (!p) return fail(E_ARG, "null params");
    memset(p, 0, sizeof *p);
    // layer list: yolo_forward.c:1202-1262 / slim_yolo_v2.py:58-87
    static const int L[10][4] = { {3, 16, 1, 1}, {16, 32, 1, 1}, {32, 64, 1, 0}, {64, 64, 1, 1}, {64, 128, 1, 0},
                                  {128, 128, 1, 1}, {128, 256, 1, 0}, {256, 256, 1, 0}, {256, 256, 1, 0}, {256, 35, 0, 0} };
    // tables: yolo_forward.c:32-35 (scale_a[0]: the literal 65536 does not fit `const char` and is stored as 0)
    static const int sw[10] = { 6, 8, 8, 9, 9, 9, 10, 10, 10, 9 };
    static const int sb[10] = { 7, 6, 5, 5, 5, 6, 5, 5, 5, 10 };
    static const int sa[11] = { 0, 4, 8, 8, 8, 8, 8, 8, 8, 16, 4 };
    static const int rt[10] = { 11, 10, 10, 11, 11, 10, 11, 11, 11, 10 };
    static const float anc[5][2] = { {0.53f, 0.79f}, {1.71f, 2.36f}, {2.89f, 6.44f}, {6.33f, 3.79f}, {9.03f, 9.74f} };
    p->num_layers = 10;
    for (int l = 0; l < 10; ++l) {
        p->layers[l].cin = L[l][0]; p->layers[l].cout = L[l][1]; p->layers[l].activ = L[l][2]; p->layers[l].pool = L[l][3];
        p->scale_w[l] = sw[l]; p->scale_b[l] = sb[l]; p->retune[l] = rt[l];
    }
    for (int l = 0; l < 11; ++l) p->scale_a[l] = sa[l];
    p->contract = YOLO_B200_CONTRACT_F; p->round_mode = YOLO_B200_ROUND_RNE; p->head_mode = YOLO_B200_HEAD_PYTHON;
    p->num_anchors = 5; p->num_classes = 2; p->stride = 16;
    for (int a = 0; a < 5; ++a) { p->anchors[a][0] = anc[a][0]; p->anchors[a][1] = anc[a][1]; }
    p->conf_thresh = 0.01f; p->nms_thresh = 0.5f; p->max_det = 1024;
    return 0;
}

int yolo_b200_create(yolo_b200_ctx **out, int device)
{
    if (!out) return fail(E_ARG, "null out");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(E_CUDA, "no CUDA device (%s): this library has no CPU fallback", e == cudaSuccess ? "count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(E_ARG, "device %d out of range (%d devices)", device, ndev);
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(E_UNSUPPORTED, "device %d is sm_%d%d; kernels are built for sm_100a only", device, prop.major, prop.minor);
    CU(cudaSetDevice(device));
    yolo_b200_ctx *c = new yolo_b200_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    c->stream = c->own_stream;
    CU(cudaMalloc(&c->ovf_dev, sizeof(unsigned)));
    CU(cudaMemset(c->ovf_dev, 0, sizeof(unsigned)));
    CU(cudaMalloc(&c->stats_dev, 2 * sizeof(int)));
    CU(cudaMalloc(&c->lut_dev, 4096 * sizeof(int)));
    CU(cudaMalloc(&c->lut8_dev, 1536));
    CU(head_init());
    *out = c;
    return 0;
}

static void free_tables(ResizeTables &t)
{
    cudaFree(t.dev);
    for (int k = 0; k < 2; ++k) {
        if (t.host[k]) cudaFreeHost(t.host[k]);
        if (t.ev[k]) cudaEventDestroy(t.ev[k]);
    }
}

static void free_layers(yolo_b200_ctx *c)
{
    for (auto &l : c->layers) { l.view = nullptr; cudaFree(l.w); cudaFree(l.w_k160); cudaFree(l.wimg); cudaFree(l.wimg_tap); cudaFree(l.wimg_tap2); cudaFree(l.wimg_tap3); cudaFree(l.wimg_rp); cudaFree(l.wimg_rps); cudaFree(l.w_swz); cudaFree(l.bias_sh); cudaFree(l.out); cudaFree(l.w1); cudaFree(l.raw); cudaFree(l.cat); }
    c->layers.clear();
}

void yolo_b200_destroy(yolo_b200_ctx *c)
{
    if (!c) return;
    {
        std::lock_guard<std::mutex> g(g_default_mu);
        if (g_default_ctx == c) g_default_ctx = nullptr;
    }
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    free_layers(c);
    cudaFree(c->lut_dev); cudaFree(c->lut8_dev); cudaFree(c->ovf_dev); cudaFree(c->stats_dev); cudaFree(c->in_q);
    cudaFree(c->rs_out); free_tables(c->rs_cache); free_tables(c->rs_call);
    cudaFree(c->h_scores); cudaFree(c->h_cls); cudaFree(c->h_boxes);
    for (auto e : c->ev) cudaEventDestroy(e);
    for (auto &S : c->slots) {
        cudaFree(S.stage_in); cudaFree(S.rs_src); cudaFree(S.pred_all); cudaFree(S.d_dets); cudaFree(S.d_counts);
        free_tables(S.tabs);
        if (S.counts_pinned) cudaFreeHost(S.counts_pinned);
        for (auto e : S.ev_in) cudaEventDestroy(e);
        for (auto e : S.ev_done) cudaEventDestroy(e);
        for (auto e : S.ev_cnt) cudaEventDestroy(e);
        if (S.ev_out) cudaEventDestroy(S.ev_out);
    }
    if (c->s_in) cudaStreamDestroy(c->s_in);
    if (c->s_out) cudaStreamDestroy(c->s_out);
    if (c->s_head) cudaStreamDestroy(c->s_head);
    cudaStreamDestroy(c->own_stream);
    delete c;
}

int yolo_b200_set_stream(yolo_b200_ctx *c, void *s)
{
    if (!c) return fail(E_ARG, "null ctx");
    c->stream = s ? (cudaStream_t)s : c->own_stream;
    return 0;
}

// pixel_norm_quantize (yolo_forward.c:57-85) evaluated once per 12-bit code: mask without shifting, /255.,
// -mean, /std in the reference's float/double mix, * 2^sa, truncation toward zero.
static void build_rgb444_lut(int sa, int8_t *lut)
{
    const int mask[3] = { 0x000f, 0x00f0, 0x0f00 };
    const double mean[3] = { 0.485, 0.456, 0.406 }, sd[3] = { 0.229, 0.224, 0.225 };
    const double s = pow(2.0, (double)sa);
    for (int code = 0; code < 4096; ++code) {
        for (int ch = 0; ch < 3; ++ch) {
            float v = (float)(code & mask[ch]);
            v = (float)((double)v / 255.);
            v = (float)((double)v - mean[ch]);
            v = (float)((double)v / sd[ch]);
            double r = (double)v * s;
            int t = (int)r;                       // toward zero
            lut[code * 4 + ch] = (int8_t)t;       // same low byte as the reference's (char) conversion in range
        }
        lut[code * 4 + 3] = 0;
    }
}

// BaseTransform without the resize + a_tracker_in, per byte value and channel (see quantize.cu).  numpy evaluates
// x /= 255.; x -= mean; x /= std in float32 (data/__init__.py:44-46,50-52); the tracker rounds x * 2^sa half-to-even
// (slim_yolo_v2.py:35).  Network channel order is RGB (test.py:79), the image is BGR.
static bool build_u8_lut(int sa, uint8_t *lut)
{
    const float mean_bgr[3] = { 0.406f, 0.456f, 0.485f }, std_bgr[3] = { 0.225f, 0.224f, 0.229f };
    const float s = ldexpf(1.0f, sa);
    bool sat = false;
    for (int ch = 0; ch < 3; ++ch) {              // ch: 0 = R, 1 = G, 2 = B of the network input = BGR byte 2 - ch
        const float mean = mean_bgr[2 - ch], sd = std_bgr[2 - ch];
        for (int v = 0; v < 256; ++v) {
            volatile float x = (float)v;
            x = x / 255.0f;
            x = x - mean;
            x = x / sd;
            float q = nearbyintf(x * s);          // default rounding mode: to nearest even
            int qi = q < -128.f ? -128 : q > 127.f ? 127 : (int)q;
            lut[ch * 256 + v] = (uint8_t)(int8_t)qi;
            lut[768 + ch * 256 + v] = (q < -128.f || q > 127.f) ? 1 : 0;
            sat |= (q < -128.f || q > 127.f);
        }
    }
    return sat;
}

// Output channels a consumer of layer k sees (reorg = space-to-depth by 2) and the activation exponent of layer l's INPUT:
// the source's output exponent; a concat brings both parts to the smaller of the two (include/yolo_b200.h: concat_with).
static int seen_channels(const yolo_b200_params *p, int k) { return p->layers[k].cout * (p->layers[k].reorg ? 4 : 1); }
static int input_exponent(const yolo_b200_params *p, int l)
{
    if (l == 0) return p->scale_a[0];
    const yolo_b200_layer &L = p->layers[l];
    const int src = L.in_from ? L.in_from - 1 : l - 1;
    int e = p->scale_a[src + 1];
    if (L.concat_with && p->scale_a[L.concat_with] < e) e = p->scale_a[L.concat_with];
    return e;
}

static int host_shr_round(int x, int n, int mode)
{
    if (n <= 0) return x;
    int fl = x >> n, rem = x - (fl << n), half = 1 << (n - 1);
    if (mode == YOLO_B200_ROUND_FLOOR) return fl;
    if (mode == YOLO_B200_ROUND_HALF_UP) return fl + (rem >= half);
    if (rem != half) return fl + (rem > half);
    return fl + (fl & 1);
}

// Host-to-device copy of data that work queued afterwards on the context stream reads (weights, biases, tables): queued on
// that stream, so it lands before that work starts.  A synchronous cudaMemcpy from pageable memory may return before its
// DMA has landed, and the context's streams are non-blocking, so they would not be ordered after it.  The source may be
// reused when this returns (pageable memory is staged before the call returns).
static cudaError_t upload(yolo_b200_ctx *c, void *dst, const void *src, size_t bytes)
{
    return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream);
}

// Epilogue programme of layer l from the context's tables (set_quantize_scale, yolo_forward.c:235-254, for contract F;
// slim_yolo_v2.py:33-38 for contract P) and the pre-shifted biases; uploads the biases.
static int derive_layer(yolo_b200_ctx *c, int l)
{
    const yolo_b200_params *p = &c->prm;
    const yolo_b200_layer &L = p->layers[l];
    LayerDev &d = c->layers[l];
    LayerQ &q = d.q;
    memset(&q, 0, sizeof q);
    q.contract = p->contract; q.round_mode = p->round_mode; q.activ = L.activ; q.pool = L.pool;
    const int sa_i = input_exponent(p, l), sw = p->scale_w[l], sb = p->scale_b[l], rt = p->retune[l], sa_o = p->scale_a[l + 1];
    std::vector<int> bsh(d.cout_pad, 0);
    const int8_t *b = d.bias_host.data();
    if (p->contract == YOLO_B200_CONTRACT_F) {
        int iofs = sa_i + sw - rt, bofs = sb - rt, oofs = rt - sa_o, bdir = 0;
        q.idir = iofs < 0; q.iofs = abs(iofs);
        bdir = bofs < 0; bofs = abs(bofs);
        q.odir = oofs < 0; q.oofs = abs(oofs);
        if (q.iofs > 24 || bofs > 20 || q.oofs > 24) return fail(E_UNSUPPORTED, "layer %d: shift out of range (iofs %d bofs %d oofs %d)", l, q.iofs, bofs, q.oofs);
        for (int o = 0; o < L.cout; ++o)
            bsh[o] = bdir ? (int)b[o] * (1 << bofs) : host_shr_round(b[o], bofs, p->round_mode);
    } else if (p->contract == YOLO_B200_CONTRACT_P) {
        int ea = sa_i + sw, E = ea > sb ? ea : sb;
        q.la = E - ea; q.sh = E - sa_o;
        // |b << lb| <= 2^7 * 2^23 = 2^30 and |acc << la| < 2^27: the int32 numerator and the rounding add cannot wrap
        if (q.la > 4 || E - sb > 23 || q.sh > 24 || q.sh < -8) return fail(E_UNSUPPORTED, "layer %d: exponents out of range (la %d lb %d sh %d)", l, q.la, E - sb, q.sh);
        for (int o = 0; o < L.cout; ++o) bsh[o] = (int)b[o] * (1 << (E - sb));
    } else return fail(E_ARG, "contract %d", p->contract);
    d.bias_abs_max = 0;
    for (int o = 0; o < L.cout; ++o) d.bias_abs_max = abs(bsh[o]) > d.bias_abs_max ? abs(bsh[o]) : d.bias_abs_max;
    CU(upload(c, d.bias_sh, bsh.data(), bsh.size() * sizeof(int)));
    return 0;
}

int yolo_b200_load(yolo_b200_ctx *c, const int8_t *const *weights, const int8_t *const *biases,
                   const yolo_b200_params *p, int layout)
{
    if (!c || !weights || !biases || !p) return fail(E_ARG, "null argument");
    if (p->num_layers < 1 || p->num_layers > YOLO_B200_MAX_LAYERS) return fail(E_ARG, "num_layers %d", p->num_layers);
    if (layout < 0 || layout > 2) return fail(E_ARG, "weight layout %d", layout);
    if (p->num_anchors < 1 || p->num_anchors > YOLO_B200_MAX_ANCHORS) return fail(E_ARG, "num_anchors %d", p->num_anchors);
    if (p->num_classes < 1 || p->num_classes > 64) return fail(E_ARG, "num_classes %d", p->num_classes);
    if (p->head_mode == YOLO_B200_HEAD_C && p->num_classes != 2) return fail(E_ARG, "the C head is 2-class (yolo_forward.c:976)");
    if (p->max_det < 1) return fail(E_ARG, "max_det %d", p->max_det);
    const yolo_b200_layer &last = p->layers[p->num_layers - 1];
    if (last.cout != p->num_anchors * (5 + p->num_classes))
        return fail(E_ARG, "last layer has %d channels, head needs %d", last.cout, p->num_anchors * (5 + p->num_classes));
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    free_layers(c);
    c->loaded = false;
    c->prm = *p;
    for (int l = 0; l < p->num_layers; ++l) {
        const yolo_b200_layer &L = p->layers[l];
        if (L.cin < 1 || L.cout < 1 || L.cin > 8192 || L.cout > 4096) return fail(E_ARG, "layer %d channels %d->%d", l, L.cin, L.cout);
        const int ks = L.ksize == 0 ? 3 : L.ksize, taps = ks * ks;
        if (ks != 1 && ks != 3) return fail(E_UNSUPPORTED, "layer %d: kernel size %d (3x3 and 1x1 only)", l, ks);
        if (L.in_from < 0 || L.in_from > l || L.concat_with < 0 || L.concat_with > l) return fail(E_ARG, "layer %d: in_from / concat_with must name an earlier layer", l);
        if (l == 0 && (L.in_from || L.concat_with)) return fail(E_ARG, "layer 0 reads the network input");
        if (l > 0) {
            const int src = L.in_from ? L.in_from - 1 : l - 1;
            if (p->layers[src].reorg) return fail(E_UNSUPPORTED, "layer %d: a reorganised map can only enter through concat_with", l);
            int want = p->layers[src].cout;
            if (L.concat_with) want += seen_channels(p, L.concat_with - 1);
            if (L.cin != want) return fail(E_ARG, "layer %d cin %d != %d channels of its input", l, L.cin, want);
            if (L.concat_with && (p->layers[src].cout % 4 || seen_channels(p, L.concat_with - 1) % 4)) return fail(E_UNSUPPORTED, "layer %d: concatenated parts must be multiples of 4 channels", l);
        }
        if (l == 0 && L.cin > 4) return fail(E_UNSUPPORTED, "network input must have <= 4 channels (NHWC4)");
        if (layout == YOLO_B200_WLAYOUT_WEIGHT_H && ks != 3) return fail(E_UNSUPPORTED, "layer %d: weight.h order is defined for 3x3 layers", l);
        if (!weights[l] || !biases[l]) return fail(E_ARG, "layer %d: null weights/biases", l);
        LayerDev d;
        d.cin = L.cin; d.cout = L.cout; d.ksize = ks; d.in_from = L.in_from; d.reorg = L.reorg; d.concat_with = L.concat_with;
        d.cs_in = yolo_b200_cstride(L.cin); d.cs_out = yolo_b200_cstride(L.cout);
        d.cout_pad = (d.cs_out + 31) / 32 * 32;
        d.bias_host.assign(biases[l], biases[l] + L.cout);
        // repack to [cout_pad][9 taps][cs_in], zero padded; a 1x1 kernel is the centre tap (the 3x3 kernels and the
        // dot-product cross-check path then run it unchanged; the tensor-core 1x1 path uses the compact one-tap copy below)
        std::vector<int8_t> &wp = d.wp_host;
        wp.assign((size_t)d.cout_pad * 9 * d.cs_in, 0);
        const int8_t *w = weights[l];
        const int tm = L.cout < 32 ? L.cout : 32, tn = L.cin < 16 ? L.cin : 16;       // weight.h groups
        const int gco = (L.cout + tm - 1) / tm, gci = (L.cin + tn - 1) / tn;
        for (int o = 0; o < L.cout; ++o)
            for (int t = 0; t < taps; ++t)
                for (int i = 0; i < L.cin; ++i) {
                    size_t src;
                    if (layout == YOLO_B200_WLAYOUT_OIHW) src = ((size_t)o * L.cin + i) * taps + t;
                    else if (layout == YOLO_B200_WLAYOUT_OHWI) src = ((size_t)o * taps + t) * L.cin + i;
                    else src = ((((size_t)t * gco + o / tm) * gci + i / tn) * tm + o % tm) * tn + i % tn;
                    wp[((size_t)o * 9 + (ks == 1 ? 4 : t)) * d.cs_in + i] = w[src];
                }
        CU(cudaMalloc(&d.w, wp.size()));
        CU(upload(c, d.w, wp.data(), wp.size()));
        if (ks == 1) {
            std::vector<int8_t> w1((size_t)d.cout_pad * d.cs_in, 0);
            for (int o = 0; o < d.cout_pad; ++o) memcpy(&w1[(size_t)o * d.cs_in], &wp[((size_t)o * 9 + 4) * d.cs_in], d.cs_in);
            CU(cudaMalloc(&d.w1, w1.size()));
            CU(upload(c, d.w1, w1.data(), w1.size()));
        }
        if (d.cs_in == 16 && ks == 3) {
            std::vector<int8_t> wk((size_t)d.cout_pad * 160, 0);
            for (int o = 0; o < d.cout_pad; ++o) memcpy(&wk[(size_t)o * 160], &wp[(size_t)o * 144], 144);
            CU(cudaMalloc(&d.w_k160, wk.size()));
            CU(upload(c, d.w_k160, wk.data(), wk.size()));
        }
        if (d.cs_in >= 16 && d.cs_in <= 256 && d.cs_out <= 256 && ks == 3) {
            // conv_ws.cu: B operand as UMMA no-swizzle K-major core matrices, [n/8][kchunk][n%8][16 B].  K chunk order is
            // tap-major (chunk = tap * cs_in/16 + c).  16-channel layers pair two taps per K = 32 MMA and carry a zero
            // 10th tap; chunks 10..19 repeat the pairs with their halves swapped (for tap pairs whose second half lies
            // at the lower shared-memory address in the parity-split tile).
            const int np = d.cs_in / 16, kc = np == 1 ? 20 : 9 * np;
            std::vector<uint8_t> img((size_t)d.cs_out * kc * 16, 0);
            for (int o = 0; o < d.cs_out; ++o)
                for (int k = 0; k < kc; ++k) {
                    int tap, c;
                    if (np == 1) { int kk = k < 10 ? k : ((k - 10) ^ 1); tap = kk; c = 0; }
                    else { tap = k / np; c = k % np; }
                    if (tap >= 9) continue;
                    memcpy(&img[(((size_t)(o / 8) * kc + k) * 8 + (o % 8)) * 16], &wp[((size_t)o * 9 + tap) * d.cs_in + 16 * c], 16);
                }
            CU(cudaMalloc(&d.wimg, img.size()));
            CU(upload(c, d.wimg, img.data(), img.size()));
            if (d.cs_in == 128 || d.cs_in == 256) {
                std::vector<uint8_t> imt((size_t)d.cs_out * 9 * d.cs_in, 0);
                // chunk = (tap, 128-channel plane): [tap][plane][cs_out/8][8 K chunks][8][16 B]
                for (int tap = 0; tap < 9; ++tap)
                    for (int o = 0; o < d.cs_out; ++o)
                        for (int cc = 0; cc < np; ++cc)
                            memcpy(&imt[(((((size_t)tap * (np / 8) + cc / 8) * (d.cs_out / 8) + o / 8) * 8 + cc % 8) * 8 + (o % 8)) * 16],
                                   &wp[((size_t)o * 9 + tap) * d.cs_in + 16 * cc], 16);
                CU(cudaMalloc(&d.wimg_tap, imt.size()));
                CU(upload(c, d.wimg_tap, imt.data(), imt.size()));
                if (d.cs_out == 256) {
                    // conv_wsp.cu: chunk = (half of the output channels, 128-channel plane, tap): [half][plane][tap][128/8][8 K chunks][8][16 B]
                    std::vector<uint8_t> im2(imt.size(), 0);
                    const int npl = np / 8;
                    for (int nh = 0; nh < 2; ++nh)
                        for (int pl = 0; pl < npl; ++pl)
                            for (int tap = 0; tap < 9; ++tap)
                                for (int o = 0; o < 128; ++o)
                                    for (int cc = 0; cc < 8; ++cc)
                                        memcpy(&im2[((((size_t)(nh * npl + pl) * 9 + tap) * 16 + o / 8) * 8 + cc) * 128 + (size_t)(o % 8) * 16],
                                               &wp[((size_t)(nh * 128 + o) * 9 + tap) * d.cs_in + pl * 128 + 16 * cc], 16);
                    CU(cudaMalloc(&d.wimg_tap2, im2.size()));
                    CU(upload(c, d.wimg_tap2, im2.data(), im2.size()));
                }
            }
        }
        if (d.cs_in == 16 && d.cs_out == 32 && ks == 3 && L.pool) {
            // conv_rp.cu: GEMM column n = dy * 32 + co (output row 2Y + dy), K chunk = (input row khh = 0..3 of 2Y-1 .. 2Y+2, tap kw):
            // the weights of tap (kh = khh - dy, kw), zero where kh falls outside 0..2.  [n/8][chunk][n%8][16 B]
            std::vector<uint8_t> img((size_t)64 * 12 * 16, 0);
            for (int dy = 0; dy < 2; ++dy)
                for (int o = 0; o < 32; ++o)
                    for (int khh = 0; khh < 4; ++khh)
                        for (int kw = 0; kw < 3; ++kw) {
                            const int kh = khh - dy, n = dy * 32 + o;
                            if (kh < 0 || kh > 2) continue;
                            memcpy(&img[(((size_t)(n / 8) * 12 + khh * 3 + kw) * 8 + (n % 8)) * 16], &wp[((size_t)o * 9 + kh * 3 + kw) * 16], 16);
                        }
            CU(cudaMalloc(&d.wimg_rp, img.size()));
            CU(upload(c, d.wimg_rp, img.data(), img.size()));
            // x-split variant: chunks 2r, 2r+1 = (input row r, kw 0), (r, kw 2); chunks 8 + r = (r, kw 1)
            std::vector<uint8_t> ims((size_t)64 * 12 * 16, 0);
            for (int dy = 0; dy < 2; ++dy)
                for (int o = 0; o < 32; ++o)
                    for (int khh = 0; khh < 4; ++khh)
                        for (int kw = 0; kw < 3; ++kw) {
                            const int kh = khh - dy, n = dy * 32 + o;
                            if (kh < 0 || kh > 2) continue;
                            const int chunk = kw == 1 ? 8 + khh : 2 * khh + (kw >> 1);
                            memcpy(&ims[(((size_t)(n / 8) * 12 + chunk) * 8 + (n % 8)) * 16], &wp[((size_t)o * 9 + kh * 3 + kw) * 16], 16);
                        }
            CU(cudaMalloc(&d.wimg_rps, ims.size()));
            CU(upload(c, d.wimg_rps, ims.data(), ims.size()));
        }
        if (ks == 3 && d.cs_in % 128 == 0 && d.cs_out % 256 == 0 && (d.cs_in > 256 || d.cs_out > 256)) {
            // conv_ws3.cu: chunk = (slice of 256 output channels, half of the slice, 128-channel plane, tap): [128/8][8 K chunks][8][16 B]
            const int npl = d.cs_in / 128, nsl = d.cs_out / 256;
            std::vector<uint8_t> im3((size_t)d.cs_out * 9 * d.cs_in, 0);
            for (int sl = 0; sl < nsl; ++sl)
                for (int hf = 0; hf < 2; ++hf)
                    for (int pl = 0; pl < npl; ++pl)
                        for (int tap = 0; tap < 9; ++tap)
                            for (int o = 0; o < 128; ++o)
                                for (int cc = 0; cc < 8; ++cc)
                                    memcpy(&im3[((((((size_t)(sl * 2 + hf) * npl + pl) * 9 + tap) * 16 + o / 8) * 8 + cc) * 8 + (o % 8)) * 16],
                                           &wp[((size_t)(sl * 256 + hf * 128 + o) * 9 + tap) * d.cs_in + pl * 128 + 16 * cc], 16);
            CU(cudaMalloc(&d.wimg_tap3, im3.size()));
            CU(upload(c, d.wimg_tap3, im3.data(), im3.size()));
        }
        // (the 128B-swizzled image of conv_umma.cu is built on first use: ensure_swz)
        CU(cudaMalloc(&d.bias_sh, (size_t)d.cout_pad * sizeof(int)));
        c->layers.push_back(d);
        { int rc = derive_layer(c, l); if (rc) return rc; }
    }
    c->graph = false;
    for (int l = 0; l < p->num_layers; ++l) {
        const yolo_b200_layer &L = p->layers[l];
        if (L.ksize == 1 || L.in_from || L.reorg || L.concat_with) c->graph = true;
        if (L.in_from && p->layers[L.in_from - 1].pool) c->layers[L.in_from - 1].unfused_pool = true;    // a route reads the un-pooled map
        if (L.pool && yolo_b200_cstride(L.cout) > 256) c->layers[l].unfused_pool = true;                 // sliced wide layers do not fuse the pool
    }
    CU(cudaMemset(c->ovf_dev, 0, sizeof(unsigned)));      // the saturation counter belongs to the loaded network
    build_rgb444_lut(p->scale_a[0], c->lut_host);
    CU(upload(c, c->lut_dev, c->lut_host, sizeof c->lut_host));
    c->lut8_saturates = build_u8_lut(p->scale_a[0], c->lut8_host);
    CU(upload(c, c->lut8_dev, c->lut8_host, sizeof c->lut8_host));
    CU(cudaStreamSynchronize(c->stream));                  // the network is on the device, whichever stream runs next
    c->loaded = true;
    return 0;
}

int yolo_b200_set_conv_backend(yolo_b200_ctx *c, int backend)
{
    if (!c) return fail(E_ARG, "null ctx");
    if (backend < 0 || backend > 5) return fail(E_ARG, "backend %d", backend);
    c->conv_backend = backend;
    return 0;
}

int yolo_b200_set_host_chunk(yolo_b200_ctx *c, int frames)
{
    if (!c) return fail(E_ARG, "null ctx");
    if (frames < 0) return fail(E_ARG, "chunk %d", frames);
    c->host_chunk = frames;
    return 0;
}

int yolo_b200_set_thresholds(yolo_b200_ctx *c, float conf, float nms)
{
    if (!c) return fail(E_ARG, "null ctx");
    c->prm.conf_thresh = conf; c->prm.nms_thresh = nms;
    return 0;
}

int yolo_b200_rgb444_lut(yolo_b200_ctx *c, int8_t *lut)
{
    if (!c || !lut) return fail(E_ARG, "null argument");
    if (!c->loaded) return fail(E_STATE, "no network loaded");
    memcpy(lut, c->lut_host, sizeof c->lut_host);
    return 0;
}

static int ensure(void **p, size_t *cap, size_t need)
{
    if (*cap >= need) return 0;
    if (*p) cudaFree(*p);
    *p = nullptr; *cap = 0;
    cudaError_t e = cudaMalloc(p, need);
    if (e != cudaSuccess) return fail(E_NOMEM, "cudaMalloc(%zu): %s", need, cudaGetErrorString(e));
    *cap = need;
    return 0;
}

static int check_ready(yolo_b200_ctx *c, int n, int h, int w)
{
    if (!c) return fail(E_ARG, "null ctx");
    if (!c->loaded) return fail(E_STATE, "no network loaded (call yolo_b200_load)");
    if (n < 0 || h < 1 || w < 1) return fail(E_ARG, "bad shape n=%d h=%d w=%d", n, h, w);
    cudaError_t e = cudaSetDevice(c->device);
    if (e != cudaSuccess) return fail(E_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    return 0;
}

static void tick(yolo_b200_ctx *c)
{
    if (!c->timing) return;
    if (c->ev_used == (int)c->ev.size()) { cudaEvent_t e; cudaEventCreate(&e); c->ev.push_back(e); }
    cudaEventRecord(c->ev[c->ev_used++], c->stream);
}

int yolo_b200_quantize_rgb444(yolo_b200_ctx *c, const uint16_t *d_frames, int n, int h, int w, int8_t *d_nhwc4)
{
    int rc = check_ready(c, n, h, w); if (rc) return rc;
    if (n == 0) return 0;
    CU(quantize_rgb444(d_frames, (size_t)n * h * w, c->lut_dev, d_nhwc4, c->stream));
    c->launches++;
    return 0;
}

int yolo_b200_quantize_f32(yolo_b200_ctx *c, const float *d_nchw, int n, int h, int w, int8_t *d_nhwc4)
{
    int rc = check_ready(c, n, h, w); if (rc) return rc;
    if (n == 0) return 0;
    if (((size_t)h * w) % 4) return fail(E_UNSUPPORTED, "h*w must be a multiple of 4");
    if (((uintptr_t)d_nchw | (uintptr_t)d_nhwc4) & 15) return fail(E_ARG, "fp32 front end: device buffers must be 16-byte aligned");
    CU(quantize_f32(d_nchw, n, h, w, c->prm.scale_a[0], d_nhwc4, c->ovf_dev, c->stream));
    c->launches++;
    return 0;
}

int yolo_b200_quantize_u8bgr(yolo_b200_ctx *c, const uint8_t *d_bgr, int n, int h, int w, int8_t *d_nhwc4)
{
    int rc = check_ready(c, n, h, w); if (rc) return rc;
    if (n == 0) return 0;
    CU(quantize_u8bgr(d_bgr, (size_t)n * h * w, c->lut8_dev, d_nhwc4, c->ovf_dev, c->stream));
    c->launches++;
    return 0;
}

int yolo_b200_resize_taps(int src, int dst, int horizontal, int32_t *taps)
{
    if (src < 1 || dst < 1 || !taps) return fail(E_ARG, "bad resize axis %d -> %d", src, dst);
    std::vector<int4> t((size_t)dst);
    resize_axis_table(src, dst, horizontal != 0, 1, t.data());
    for (int d = 0; d < dst; ++d) { taps[4 * d] = t[d].x; taps[4 * d + 1] = t[d].y; taps[4 * d + 2] = t[d].z; taps[4 * d + 3] = t[d].w; }
    return 0;
}

static int ensure_pinned(char **p, size_t *cap, size_t need)
{
    if (*cap >= need) return 0;
    if (*p) cudaFreeHost(*p);
    *p = nullptr; *cap = 0;
    cudaError_t e = cudaHostAlloc((void **)p, need, cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(E_NOMEM, "cudaHostAlloc(%zu): %s", need, cudaGetErrorString(e));
    *cap = need;
    return 0;
}

// One frame (BGR, a YUV layout, a Bayer pattern or a pixel format) of (format, sh, sw): its packed byte count, or E_ARG /
// E_UNSUPPORTED (include/yolo_b200.h).  The formats, the sizes each accepts and their frame bytes (camera_frame_bytes) live
// here, and so does the check of a pitched layout (layout_check).  BGR and the pixel formats take any size of at least 1x1.
static int source_check(int format, int sh, int sw, size_t *bytes)
{
    const bool yuv = format == RS_YUV_NV12 || format == RS_YUV_I420 || format == RS_YUV_YUYV;
    const bool bayer = format >= RS_BAYER_RGGB && format <= RS_BAYER_BGGR;
    const bool pix = format >= RS_RGB && format <= RS_RGB_PLANAR;
    if (!yuv && !bayer && !pix && format != RS_BGR) return fail(E_ARG, "unknown source format %d", format);
    if (sh < 1 || sw < 1) return fail(E_ARG, "bad source shape %dx%d", sh, sw);
    if (yuv && (sw % 2 || (format != RS_YUV_YUYV && sh % 2)))
        return fail(E_ARG, "YUV format %d needs an even %s (%dx%d)", format, format == RS_YUV_YUYV ? "width" : "height and width", sh, sw);
    if (bayer && (sh < 3 || sw < 3)) return fail(E_ARG, "a Bayer frame needs at least 3x3 pixels (%dx%d)", sh, sw);
    *bytes = camera_frame_bytes(format, sh, sw);
    if (*bytes > (size_t)INT32_MAX) return fail(E_UNSUPPORTED, "camera frame larger than 2 GiB");
    return 0;
}

// The source format of a YUV entry point's format (the public codes are the internal ones), of a Bayer entry point's
// pattern and of a pixel-format entry point's format; anything else goes on as an unknown format, which source_check refuses
static int yuv_format(int format) { return format >= YOLO_B200_YUV_NV12 && format <= YOLO_B200_YUV_YUYV ? format : -1; }
static int pix_format(int format) { return format >= YOLO_B200_PIX_RGB && format <= YOLO_B200_PIX_RGB_PLANAR ? RS_RGB + format : -1; }
static int bayer_format(int pattern)
{
    static const int fmt[4] = { RS_BAYER_RGGB, RS_BAYER_BGGR, RS_BAYER_GRBG, RS_BAYER_GBRG };     // YOLO_B200_BAYER_* order
    static_assert(YOLO_B200_BAYER_RGGB == 0 && YOLO_B200_BAYER_BGGR == 1 && YOLO_B200_BAYER_GRBG == 2 && YOLO_B200_BAYER_GBRG == 3, "pattern codes");
    return pattern >= 0 && pattern < 4 ? fmt[pattern] : -1;
}
// The source format of a frames descriptor's (family, format)
static int family_format(int family, int format)
{
    switch (family) {
    case YOLO_B200_SRC_BGR:   return RS_BGR;
    case YOLO_B200_SRC_YUV:   return yuv_format(format);
    case YOLO_B200_SRC_BAYER: return bayer_format(format);
    case YOLO_B200_SRC_PIX:   return pix_format(format);
    default:                  return -1;
    }
}

// A pitched layout of frames of (format, sh, sw), already checked by source_check: where one frame's planes start
// relative to the frame and how far they reach.  Every plane the format has needs offset >= 0 and a pitch of at least its
// row bytes (E_ARG; planes it lacks are ignored), the stride >= 0 (E_ARG; frames may overlap, the source is read only);
// a frame spanning more than 2 GiB is E_UNSUPPORTED.  *first / *end: the frame's span [first, end) from its start.
static int layout_check(int format, const yolo_b200_frames &d, int64_t *first, int64_t *end, ResizeLayout *lay)
{
    int rows[3], row_bytes[3];
    const int planes = source_planes(format, d.sh, d.sw, rows, row_bytes);
    if (d.frame_stride < 0) return fail(E_ARG, "negative frame stride %lld", (long long)d.frame_stride);
    constexpr int64_t FAR = (int64_t)1 << 62;                       // keeps the sums below exact; nothing real is so far
    int64_t lo = INT64_MAX, hi = 0;
    for (int p = 0; p < planes; ++p) {
        const int64_t off = d.plane_offset[p], pitch = d.row_pitch[p];
        if (off < 0) return fail(E_ARG, "plane %d: negative offset %lld", p, (long long)off);
        if (pitch < row_bytes[p]) return fail(E_ARG, "plane %d: row pitch %lld below the %d bytes of a row", p, (long long)pitch, row_bytes[p]);
        if (off > FAR || d.frame_stride > FAR || (rows[p] > 1 && pitch > INT32_MAX))
            return fail(E_UNSUPPORTED, "plane %d: a frame larger than 2 GiB", p);
        lo = std::min(lo, off);
        hi = std::max(hi, off + (int64_t)(rows[p] - 1) * pitch + row_bytes[p]);
    }
    if (hi - lo > INT32_MAX) return fail(E_UNSUPPORTED, "a frame spans %lld bytes, more than 2 GiB", (long long)(hi - lo));
    *first = lo; *end = hi;
    if (lay) {
        *lay = ResizeLayout{};
        lay->stride = (unsigned long long)d.frame_stride;
        for (int p = 0; p < planes; ++p) {
            lay->off[p] = (unsigned)(d.plane_offset[p] - lo);
            lay->pitch[p] = rows[p] > 1 ? (unsigned)d.row_pitch[p] : (unsigned)row_bytes[p];     // one row: its pitch is never used
        }
    }
    return 0;
}

int yolo_b200_frames_packed(yolo_b200_frames *d, int family, int format, int sh, int sw)
{
    if (!d) return fail(E_ARG, "null descriptor");
    const int fmt = family_format(family, format);
    size_t bytes = 0;
    int rc = source_check(fmt, sh, sw, &bytes); if (rc) return rc;
    int rows[3], row_bytes[3];
    const int planes = source_planes(fmt, sh, sw, rows, row_bytes);
    yolo_b200_frames f{};
    f.family = family; f.format = family == YOLO_B200_SRC_BGR ? 0 : format; f.sh = sh; f.sw = sw;
    f.frame_stride = (int64_t)bytes;
    for (int p = 0, off = 0; p < planes; off += rows[p] * row_bytes[p], ++p) { f.plane_offset[p] = off; f.row_pitch[p] = row_bytes[p]; }
    *d = f;
    return 0;
}

int yolo_b200_frames_span(const yolo_b200_frames *d, int n, int64_t *first, int64_t *end)
{
    if (!d || !first || !end) return fail(E_ARG, "null argument");
    if (n < 0) return fail(E_ARG, "n %d", n);
    const int fmt = family_format(d->family, d->format);
    size_t bytes = 0;
    int rc = source_check(fmt, d->sh, d->sw, &bytes); if (rc) return rc;
    int64_t lo = 0, hi = 0;
    rc = layout_check(fmt, *d, &lo, &hi, nullptr); if (rc) return rc;
    if (n == 0) { *first = *end = 0; return 0; }
    if (n > 1 && d->frame_stride > (INT64_MAX - hi) / (n - 1)) return fail(E_UNSUPPORTED, "the frames span more than 2^63 bytes");
    *first = lo; *end = (int64_t)(n - 1) * d->frame_stride + hi;
    return 0;
}

int yolo_b200_yuv_frame_bytes(int format, int sh, int sw)
{
    size_t b = 0;
    int rc = source_check(yuv_format(format), sh, sw, &b); if (rc) return rc;
    return (int)b;
}

int yolo_b200_pix_frame_bytes(int format, int sh, int sw)
{
    size_t b = 0;
    int rc = source_check(pix_format(format), sh, sw, &b); if (rc) return rc;
    return (int)b;
}

// Where the n frames of one call are and how they become dh x dw frames of the network input (plan_sources, net_plan).
enum { RESIZE_NONE, RESIZE_UNIFORM, RESIZE_RAGGED };
struct SourcePlan {
    InKind kind = IN_BGR;                            // what the frames are once resized
    int fmt = RS_BGR, n = 0, dh = 0, dw = 0, mode = RESIZE_NONE;
    size_t frame_bytes = 0;                          // one source size: bytes per frame (pitched: the frame stride)
    std::vector<size_t> off;                         // RESIZE_RAGGED: [n + 1] byte offset of frame f; off[n] = total
    std::vector<ResizeFrame> frames;                 // RESIZE_RAGGED: what the kernel reads per frame
    std::vector<std::pair<int, int>> geoms;          // distinct source sizes in order of first appearance
    bool pitched = false;                            // a yolo_b200_frames layout (uniform): lay, and a frame's span
    ResizeLayout lay{};                              // [first, last) from its start
    size_t first = 0, last = 0;
    size_t at(int f) const { return off.empty() ? (size_t)f * frame_bytes : off[f]; }     // byte offset of frame f
    size_t begin(int f) const { return at(f) + first; }                                  // first byte frames f.. read
    size_t end(int f0, int nf) const { return pitched ? at(f0 + nf - 1) + last : at(f0 + nf); }   // one past frames [f0, f0 + nf)
};

// The plan of n frames of format fmt (RS_BGR or a camera format) for the network size dh x dw.  Frame i has the source size
// src_hw[2 * i * stride] x src_hw[2 * i * stride + 1] (stride 0: one size for all, checked also when n == 0).  One rule
// picks the resize: none for a forward call whose only source size is dh x dw in BGR (the frames are the network input
// as they are), uniform for one source size or any camera-format call, ragged for several source sizes.
// layout (one size, src_hw = its size): the frames are pitched as it says, and are resized even at the network size.
static int plan_sources(int fmt, int n, const int32_t *src_hw, int stride, int dh, int dw, bool forward, SourcePlan &p,
                        const yolo_b200_frames *layout = nullptr)
{
    p = SourcePlan();
    p.fmt = fmt; p.n = n; p.dh = dh; p.dw = dw;
    const int m = stride ? n : 1;                                // sizes to read
    if (m > 0 && !src_hw) return fail(E_ARG, "null src_hw");
    if (fmt != RS_BGR || layout) {
        int rc = source_check(fmt, src_hw[0], src_hw[1], &p.frame_bytes); if (rc) return rc;
        p.geoms.push_back({src_hw[0], src_hw[1]});
        p.mode = RESIZE_UNIFORM;
        if (!layout) return 0;
        int64_t first = 0, last = 0;
        rc = layout_check(fmt, *layout, &first, &last, &p.lay); if (rc) return rc;
        p.pitched = true; p.frame_bytes = (size_t)layout->frame_stride; p.first = (size_t)first; p.last = (size_t)last;
        return 0;
    }
    p.off.assign((size_t)(m > 0 ? m : 0) + 1, 0);
    std::map<std::pair<int, int>, int> index;
    for (int i = 0; i < m; ++i) {
        const int sh = src_hw[2 * (size_t)i], sw = src_hw[2 * (size_t)i + 1];
        if (sh < 1 || sw < 1) return fail(E_ARG, "image %d: bad source shape %dx%d", i, sh, sw);
        const size_t bytes = (size_t)sh * sw * 3;
        if (bytes > (size_t)INT32_MAX) return fail(E_UNSUPPORTED, "image %d: source image larger than 2 GiB", i);
        auto it = index.emplace(std::make_pair(sh, sw), (int)p.geoms.size()).first;
        if (it->second == (int)p.geoms.size()) p.geoms.push_back(it->first);
        p.frames.push_back({p.off[i], sw * 3, it->second});
        p.off[i + 1] = p.off[i] + bytes;
    }
    if (p.geoms.size() > 1) { p.mode = RESIZE_RAGGED; return 0; }
    p.off.clear(); p.frames.clear();
    if (p.geoms.empty()) return 0;                               // no frames
    p.frame_bytes = (size_t)p.geoms[0].first * p.geoms[0].second * 3;
    p.mode = forward && p.geoms[0] == std::make_pair(dh, dw) ? RESIZE_NONE : RESIZE_UNIFORM;
    return 0;
}

// n frames of kind k at the network size h x w: no resize, frame f at f * h * w * (bytes per pixel)
static SourcePlan net_plan(InKind k, int n, int h, int w)
{
    static const size_t px_bytes[4] = { 4, 2, 3, 12 };           // IN_INT8, IN_RGB444, IN_BGR, IN_F32
    SourcePlan p;
    p.kind = k; p.n = n; p.dh = h; p.dw = w; p.frame_bytes = (size_t)h * w * px_bytes[k];
    return p;
}

// Copies the table image img to t.dev in stream order on st: after everything queued there before it, and out of a staging
// buffer that is refilled only once the copy out of it two uploads ago has run.
static int upload_tables(ResizeTables &t, const void *img, size_t bytes, cudaStream_t st)
{
    const int k = t.next;
    if (!t.ev[k]) CU(cudaEventCreateWithFlags(&t.ev[k], cudaEventDisableTiming));
    CU(cudaEventSynchronize(t.ev[k]));
    int rc = ensure_pinned(&t.host[k], &t.host_cap[k], bytes); if (rc) return rc;
    rc = ensure(&t.dev, &t.dev_cap, bytes); if (rc) return rc;      // (a cudaFree waits for queued work)
    memcpy(t.host[k], img, bytes);
    CU(cudaMemcpyAsync(t.dev, t.host[k], bytes, cudaMemcpyHostToDevice, st));
    CU(cudaEventRecord(t.ev[k], st));
    t.next ^= 1;
    return 0;
}

// The tables the resize of plan p reads (*out; nothing for mode none).  One source size: the context's cache, uploaded on
// the context stream when the geometry changes.  Several: the descriptors, then per distinct size exactly the uniform
// tables, uploaded into `call` on stream st.
static int resize_tables(yolo_b200_ctx *c, const SourcePlan &p, ResizeTables &call, cudaStream_t st, const ResizeTables **out)
{
    if (p.mode == RESIZE_NONE) return 0;
    const bool ragged = p.mode == RESIZE_RAGGED;
    ResizeTables &t = ragged ? call : c->rs_cache;
    *out = &t;
    // a pitched plan's layout record leads the image (the kernel reads it through `frames`) and is part of the key
    const long long key[10] = { p.geoms[0].first, p.geoms[0].second, p.dh, p.dw, p.pitched, (long long)p.lay.stride,
                                p.lay.off[0] | (long long)p.lay.pitch[0] << 32, p.lay.off[1] | (long long)p.lay.pitch[1] << 32,
                                p.lay.off[2] | (long long)p.lay.pitch[2] << 32, 0 };
    if (!ragged && !memcmp(t.key, key, sizeof key)) return 0;
    const size_t G = p.geoms.size(), head = p.pitched ? sizeof(ResizeLayout) : p.frames.size() * sizeof(ResizeFrame);
    const size_t ytab_off = head, xtab_off = ytab_off + G * p.dh * sizeof(int4);
    const size_t bytes = xtab_off + G * p.dw * sizeof(int2);
    std::vector<int4> img((bytes + sizeof(int4) - 1) / sizeof(int4));
    char *b = reinterpret_cast<char *>(img.data());
    if (p.pitched) memcpy(b, &p.lay, head);
    else memcpy(b, p.frames.data(), head);
    for (size_t g = 0; g < G; ++g)
        resize_geometry_tables(p.geoms[g].first, p.geoms[g].second, p.dh, p.dw, reinterpret_cast<int4 *>(b + ytab_off) + g * p.dh,
                               reinterpret_cast<int2 *>(b + xtab_off) + g * p.dw);
    t.key[0] = 0;
    int rc = upload_tables(t, img.data(), bytes, ragged ? st : c->stream); if (rc) return rc;
    if (!ragged) memcpy(t.key, key, sizeof key);
    const char *d = (const char *)t.dev;
    t.frames = (const ResizeFrame *)d; t.ytab = (const int4 *)(d + ytab_off); t.xtab = (const int2 *)(d + xtab_off);
    return 0;
}

// One resize launch on the context stream: frames [f0, f0 + nf) of plan p (src = where byte p.begin(0) is: frame 0's start,
// or the first byte of its span when pitched) into dst.  A ragged launch may read up to the end of frame f0 + nf - 1 (in the
// host path the end of the chunk's landed bytes, never into a later chunk); a uniform one reads only its own frames, a
// pitched one only the span of its frames, p.begin(f0) .. p.end(f0, nf).
static cudaError_t enqueue_resize(yolo_b200_ctx *c, const SourcePlan &p, const ResizeTables &t, const uint8_t *src, int f0, int nf, uint8_t *dst)
{
    const bool ragged = p.mode == RESIZE_RAGGED;
    const size_t first = ragged ? 0 : p.at(f0);
    const bool words = p.lay.stride % 4 == 0 && p.lay.pitch[0] % 4 == 0;
    cudaError_t e = resize_u8c3(src + first, p.end(f0, nf) - p.first - first, p.fmt, ragged ? t.frames + f0 : nullptr, nf, p.geoms[0].first,
                                p.geoms[0].second, dst, p.dh, p.dw, t.xtab, t.ytab, c->sm_count, c->stream,
                                p.pitched ? reinterpret_cast<const ResizeLayout *>(t.frames) : nullptr, words);
    if (e == cudaSuccess) c->launches++;
    return e;
}

// The resize of the device entry points: tables, then one launch, both on the context stream
static int resize_dev(yolo_b200_ctx *c, const SourcePlan &p, const uint8_t *d_src, uint8_t *d_dst)
{
    const ResizeTables *t = nullptr;
    int rc = resize_tables(c, p, c->rs_call, c->stream, &t); if (rc) return rc;
    CU(enqueue_resize(c, p, *t, d_src + p.first, 0, p.n, d_dst));
    return 0;
}

// The resize stages: n frames (sizes as plan_sources reads them) -> uint8 BGR [n][dh][dw][3], one launch when n >= 1
static int resize_stage(yolo_b200_ctx *c, int fmt, const uint8_t *d_src, int n, const int32_t *src_hw, int stride, uint8_t *d_dst, int dh, int dw,
                        const yolo_b200_frames *layout = nullptr)
{
    if (!c) return fail(E_ARG, "null ctx");
    if (n < 0 || dh < 1 || dw < 1) return fail(E_ARG, "bad resize shape n=%d -> %dx%d", n, dh, dw);
    SourcePlan p;
    int rc = plan_sources(fmt, n, src_hw, stride, dh, dw, false, p, layout); if (rc) return rc;
    CU(cudaSetDevice(c->device));
    if (n == 0) return 0;
    if (!d_src || !d_dst) return fail(E_ARG, "null buffer");
    return resize_dev(c, p, d_src, d_dst);
}

int yolo_b200_resize_u8bgr(yolo_b200_ctx *c, const uint8_t *d_src, int n, int sh, int sw, uint8_t *d_dst, int dh, int dw)
{
    const int32_t hw[2] = { sh, sw };
    return resize_stage(c, RS_BGR, d_src, n, hw, 0, d_dst, dh, dw);
}

int yolo_b200_resize_u8bgr_ragged(yolo_b200_ctx *c, const uint8_t *d_src, int n, const int32_t *src_hw, uint8_t *d_dst, int dh, int dw)
{ return resize_stage(c, RS_BGR, d_src, n, src_hw, 1, d_dst, dh, dw); }

int yolo_b200_yuv_to_bgr_resize(yolo_b200_ctx *c, const uint8_t *d_src, int format, int n, int sh, int sw, uint8_t *d_dst, int dh, int dw)
{
    const int32_t hw[2] = { sh, sw };
    return resize_stage(c, yuv_format(format), d_src, n, hw, 0, d_dst, dh, dw);
}

int yolo_b200_bayer_to_bgr_resize(yolo_b200_ctx *c, const uint8_t *d_src, int pattern, int n, int sh, int sw, uint8_t *d_dst, int dh, int dw)
{
    const int32_t hw[2] = { sh, sw };
    return resize_stage(c, bayer_format(pattern), d_src, n, hw, 0, d_dst, dh, dw);
}

int yolo_b200_pix_to_bgr_resize(yolo_b200_ctx *c, const uint8_t *d_src, int format, int n, int sh, int sw, uint8_t *d_dst, int dh, int dw)
{
    const int32_t hw[2] = { sh, sw };
    return resize_stage(c, pix_format(format), d_src, n, hw, 0, d_dst, dh, dw);
}

// The calls on a frames descriptor: its format and size, then the family's path with the layout
#define YB_FRAMES(d) if (!(d)) return fail(E_ARG, "null frames descriptor"); const int32_t hw[2] = { (d)->sh, (d)->sw }; const int fmt = family_format((d)->family, (d)->format)

int yolo_b200_frames_to_bgr_resize(yolo_b200_ctx *c, const uint8_t *d_src, const yolo_b200_frames *d, int n, uint8_t *d_dst, int dh, int dw)
{
    YB_FRAMES(d);
    return resize_stage(c, fmt, d_src, n, hw, 0, d_dst, dh, dw, d);
}

int yolo_b200_u8bgr_lut(yolo_b200_ctx *c, int8_t *lut_host)
{
    if (!c || !lut_host) return fail(E_ARG, "null argument");
    if (!c->loaded) return fail(E_STATE, "no network loaded");
    memcpy(lut_host, c->lut8_host, 768);
    return 0;
}

// conv_umma.cu's B operand: block kb = (tap, 128-byte channel chunk) as it must sit in shared memory for a K-major
// SWIZZLE_128B operand: row r (output channel) is 128 bytes, its 16-byte chunk c lives at chunk c ^ (r & 7).  Built on first use:
// the layers the weight-stationary kernel takes never need it.
static int ensure_swz(yolo_b200_ctx *c, LayerDev &d)
{
    if (d.w_swz || d.cs_in % 128) return 0;
    const int taps = d.ksize == 1 ? 1 : 9, per = d.cs_in / 128, nkb = taps * per;
    std::vector<uint8_t> sw((size_t)nkb * d.cs_out * 128, 0);
    for (int kb = 0; kb < nkb; ++kb) {
        const int tap = d.ksize == 1 ? 4 : kb / per, c0 = (kb % per) * 128;
        for (int r = 0; r < d.cs_out; ++r)
            for (int ch = 0; ch < 8; ++ch)
                memcpy(&sw[((size_t)kb * d.cs_out + r) * 128 + (size_t)((ch ^ (r & 7)) * 16)],
                       &d.wp_host[((size_t)r * 9 + tap) * d.cs_in + c0 + 16 * ch], 16);
    }
    CU(cudaSetDevice(c->device));
    CU(cudaMalloc(&d.w_swz, sw.size()));
    CU(upload(c, d.w_swz, sw.data(), sw.size()));
    return 0;
}

static void fill_args(yolo_b200_ctx *c, int l, const int8_t *d_in, int n, int h, int w, int8_t *d_out, ConvArgs &a)
{
    LayerDev &L = c->layers[l];
    a.in = d_in; a.n = n; a.H = h; a.W = w; a.cs_in = L.cs_in; a.wgt = L.w; a.bias_sh = L.bias_sh;
    a.cout = L.cout; a.cs_out = L.cs_out; a.q = L.q; a.out = d_out; a.ovf = c->ovf_dev;
    a.wgt_k160 = L.w_k160; a.wimg = L.wimg; a.wimg_tap = L.wimg_tap; a.wimg_tap2 = L.wimg_tap2; a.wimg_tap3 = L.wimg_tap3; a.wimg_rp = L.wimg_rp; a.wimg_rps = L.wimg_rps; a.w_rows = L.cout_pad; a.bias_abs_max = L.bias_abs_max;
    a.wgt_swz = L.w_swz; a.wgt_swz_rows = L.cs_out;
    a.taps = 9; a.wgt1 = nullptr;
    a.force_generic_epilogue = c->conv_backend == 3 || c->conv_backend == 5;
}

// Layer l's output map may be stored with its rows split by x parity when the kernel that produces it can write that layout
// (the first-layer kernel, pooled, 16 channels) and its only reader, layer l + 1, runs on the row-pair kernel's x-split variant
// (conv_rp.cu).  (oh, ow) = layer l's output size.  The layout is private to the chain: yolo_b200_get_layer_output undoes it.
static bool want_xsplit(yolo_b200_ctx *c, size_t l, const void *d_in0, int n, int oh, int ow)
{
    if (c->conv_backend != 0 || c->graph || l != 0 || c->layers.size() < 2 || n < 1) return false;
    LayerDev &L = c->layers[0];
    if (!L.q.pool || L.cs_out != 16 || (ow & 1) || L.unfused_pool) return false;
    (void)d_in0;
    ConvArgs a1;
    fill_args(c, 1, L.out, n, oh, ow, c->layers[1].out, a1);
    a1.in = (const int8_t *)nullptr; a1.out = nullptr;             // alignment of the real buffers: cudaMalloc'ed, 256-byte aligned
    return conv3x3_rp_split_supported(a1);
}

// One convolution launch.  fuse_pool == false runs a pooled layer WITHOUT its pool (the caller pools separately).
static int run_layer(yolo_b200_ctx *c, int l, const int8_t *d_in, int n, int h, int w, int8_t *d_out, bool fuse_pool = true,
                     bool in_xsplit = false, bool out_xsplit = false)
{
    LayerDev &L = c->layers[l];
    ConvArgs a;
    fill_args(c, l, d_in, n, h, w, d_out, a);
    if (!fuse_pool) a.q.pool = 0;
    a.in_xsplit = in_xsplit; a.out_xsplit = out_xsplit;
    if (in_xsplit) {                     // only the row-pair kernel reads that layout (want_xsplit checked that it takes this layer)
        if (c->conv_backend != 0 || !conv3x3_rp_split_supported(a)) return fail(E_STATE, "layer %d cannot read an x-split map", l);
        CU(conv3x3_rp(a, c->stream, c->sm_count));
        c->launches++;
        return 0;
    }
    const bool aligned = (((uintptr_t)d_in | (uintptr_t)d_out) & 15) == 0;
    const int be = c->conv_backend;
    if (L.ksize == 1 || L.cs_in > 256 || L.cs_out > 256) {
        // yolo_v2 / darknet19 shapes: 1x1 layers and layers wider than 256 channels run on the streaming tcgen05 implicit GEMM
        // (one K block per (tap, 128-channel chunk), output channels in slices of 256); back end 1 keeps the dot-product kernel
        ConvArgs u = a;
        if (L.ksize == 1) { u.taps = 1; u.wgt1 = L.w1; }
        if (be == 0 && L.ksize == 3 && aligned && conv3x3_ws3_supported(a, c->sm_count)) {
            CU(conv3x3_ws3(a, c->stream, c->sm_count));        // wide 3x3 layer on a narrow map: the CTA-pair kernel
        } else if (be != 1 && aligned && conv3x3_umma_supported(u)) {
            int rc = ensure_swz(c, L); if (rc) return rc;
            u.wgt_swz = L.w_swz;
            CU(conv3x3_umma(u, c->stream, c->sm_count));
        } else {
            if (be != 0 && be != 1) return fail(E_UNSUPPORTED, "layer %d has no tensor-core shape (cs_in %d, cs_out %d, %dx%d)", l, L.cs_in, L.cs_out, L.ksize, L.ksize);
            if (be == 0) c->slow_path_launches++;
            CU(conv3x3_direct(a, c->stream));              // (a 1x1 layer is the centre tap of the 9-tap weights)
        }
        c->launches++;
        return 0;
    }
    bool umma_ok = aligned && conv3x3_umma_supported(a);
    const bool ws_ok = aligned && conv3x3_ws_supported(a);
    if ((be == 2 || be == 3) && !umma_ok) return fail(E_UNSUPPORTED, "layer %d has no tensor-core shape (cs_in %d, cs_out %d)", l, L.cs_in, L.cs_out);
    if ((be == 4 || be == 5) && !ws_ok) return fail(E_UNSUPPORTED, "layer %d does not fit the weight-stationary kernel (cs_in %d, cs_out %d)", l, L.cs_in, L.cs_out);
    const bool first_ok = ((uintptr_t)d_out & 3) == 0 && conv3x3_first_src_ok(IN_INT8, d_in) && conv3x3_first_supported(a);
    const bool use_umma = be == 2 || be == 3 || (be == 0 && !first_ok && !ws_ok && umma_ok);
    if (use_umma) { int rc = ensure_swz(c, L); if (rc) return rc; a.wgt_swz = L.w_swz; }
    if (be == 1) CU(conv3x3_direct(a, c->stream));
    else if (be == 0 && first_ok) { CU(conv3x3_first(a, c->stream)); c->launches += conv3x3_fs_supported(a, IN_INT8, a.in) ? 0 : L.cs_out / 16 - 1; }   // conv_first.cu: one pass per 16 output channels
    else if (use_umma) CU(conv3x3_umma(a, c->stream, c->sm_count));
    else if (be == 0 && conv3x3_rp_supported(a)) CU(conv3x3_rp(a, c->stream, c->sm_count));
    else if (be == 0 && aligned && conv3x3_ws2_supported(a, c->sm_count)) CU(conv3x3_ws2(a, c->stream, c->sm_count));
    else if (be == 0 && aligned && conv3x3_wsp_supported(a)) CU(conv3x3_wsp(a, c->stream, c->sm_count));
    else if (be == 4 || be == 5 || ws_ok) CU(conv3x3_ws(a, c->stream, c->sm_count));
    else {
        // auto back end, no tensor-core kernel takes this shape / alignment (e.g. a first layer wider than 16 channels, a
        // 2-byte-aligned buffer): the dot-product kernel computes the same values; counted, see yolo_b200_slow_path_count
        if (be == 0) c->slow_path_launches++;
        CU(conv3x3_direct(a, c->stream));
    }
    c->launches++;
    return 0;
}

int yolo_b200_debug_requant(yolo_b200_ctx *c, int layer, const int32_t *d_acc, size_t count, int8_t *d_out, int force_generic)
{
    int rc = check_ready(c, 0, 1, 1); if (rc) return rc;
    if (layer < 0 || layer >= (int)c->layers.size()) return fail(E_ARG, "layer %d out of range", layer);
    if ((!d_acc || !d_out) && count) return fail(E_ARG, "null buffer");
    LayerDev &L = c->layers[layer];
    ConvArgs a;
    memset(&a, 0, sizeof a);
    a.cout = L.cout; a.cs_out = L.cs_out; a.q = L.q; a.bias_sh = L.bias_sh; a.bias_abs_max = L.bias_abs_max;
    a.force_generic_epilogue = force_generic;
    int epi = 0;
    CU(requant_probe(a, d_acc, count, d_out, &epi, c->stream));
    c->launches++;
    return epi;
}

int yolo_b200_conv_layer(yolo_b200_ctx *c, int layer, const int8_t *d_in, int n, int h, int w, int8_t *d_out)
{
    int rc = check_ready(c, n, h, w); if (rc) return rc;
    if (layer < 0 || layer >= (int)c->layers.size()) return fail(E_ARG, "layer %d out of range", layer);
    if (!d_in || !d_out) return fail(E_ARG, "null buffer");
    if (n == 0) return 0;
    if (c->layers[layer].q.pool && (h < 2 || w < 2)) return fail(E_ARG, "layer %d pools: needs h,w >= 2", layer);
    return run_layer(c, layer, d_in, n, h, w, d_out);
}

// Input of layer l for this call: the previous layer's output, the un-pooled output of layer in_from - 1, or the channel
// concatenation of the two sources of a concat layer (built here by graph.cu: reorg + exponent alignment).
static int layer_input(yolo_b200_ctx *c, size_t l, const int8_t *net_in, int n, int h0, int w0, const int8_t **in, int *ih, int *iw)
{
    if (l == 0) { *in = net_in; *ih = h0; *iw = w0; return 0; }
    LayerDev &L = c->layers[l];
    const yolo_b200_params &p = c->prm;
    const int src = L.in_from ? L.in_from - 1 : (int)l - 1;
    LayerDev &S = c->layers[src];
    const int8_t *b = L.in_from ? (S.unfused_pool ? S.raw : S.view) : S.view;
    int bh = L.in_from ? S.rh : S.oh, bw = L.in_from ? S.rw : S.ow;
    if (!L.concat_with) { *in = b; *ih = bh; *iw = bw; return 0; }
    LayerDev &A = c->layers[L.concat_with - 1];
    const int ah = A.reorg ? A.oh / 2 : A.oh, aw = A.reorg ? A.ow / 2 : A.ow;
    if (ah != bh || aw != bw || (A.reorg && ((A.oh | A.ow) & 1)))
        return fail(E_ARG, "layer %zu: concatenated maps differ in size (%dx%d vs %dx%d)", l, ah, aw, bh, bw);
    int rc = ensure((void **)&L.cat, &L.cat_cap, (size_t)(n > 0 ? n : 1) * bh * bw * L.cs_in); if (rc) return rc;
    const int ea = p.scale_a[L.concat_with], eb = p.scale_a[src + 1], e = ea < eb ? ea : eb;
    if (n > 0) {
        CU(concat_reorg(A.view, A.cs_out, A.cout, A.reorg, ea - e, b, S.cs_out, S.cout, eb - e, n, bh, bw, L.cs_in, L.cat, c->stream));
        c->launches++;
    }
    *in = L.cat; *ih = bh; *iw = bw;
    return 0;
}

// Layers first..last on the context stream.  `net_in` is the network input (h x w) when first == 0; for first > 0 the
// earlier layers' outputs are already in place.
// `last_out` != nullptr: the last layer writes there instead of into its own buffer (a slot of a batch-wide prediction map).
static int backbone_from(yolo_b200_ctx *c, size_t first, const int8_t *net_in, int n, int h, int w, const int8_t **d_pred, int *gh, int *gw,
                         int8_t *last_out = nullptr)
{
    int rc;
    const int8_t *cur = net_in;
    for (size_t l = first; l < c->layers.size(); ++l) {
        LayerDev &L = c->layers[l];
        int ih, iw;
        if (l == first && first > 0 && !c->graph) { ih = h; iw = w; }                // (chain: the caller passes layer `first`'s input)
        else { rc = layer_input(c, l, net_in, n, h, w, &cur, &ih, &iw); if (rc) return rc; }
        if (L.q.pool && (ih < 2 || iw < 2)) return fail(E_ARG, "input too small: layer %zu pools a %dx%d map", l, ih, iw);
        const int oh = L.q.pool ? ih / 2 : ih, ow = L.q.pool ? iw / 2 : iw;
        int8_t *dst = L.out;
        if (last_out && l + 1 == c->layers.size()) dst = last_out;
        else {
            size_t bytes = (size_t)(n > 0 ? n : 1) * oh * ow * L.cs_out;
            rc = ensure((void **)&L.out, &L.out_cap, bytes); if (rc) return rc;
            dst = L.out;
        }
        L.oh = oh; L.ow = ow; L.rh = ih; L.rw = iw; L.view = dst;
        const bool in_split = l > 0 && !c->graph && c->layers[l - 1].xsplit;
        ConvArgs a0chk;
        fill_args(c, (int)l, cur, n, ih, iw, dst, a0chk);
        L.xsplit = l == 0 && dst == L.out && ((uintptr_t)dst & 3) == 0 && conv3x3_first_src_ok(IN_INT8, cur) && conv3x3_first_supported(a0chk) &&
                   want_xsplit(c, l, cur, n, oh, ow);
        if (L.q.pool && L.unfused_pool) {
            rc = ensure((void **)&L.raw, &L.raw_cap, (size_t)(n > 0 ? n : 1) * ih * iw * L.cs_out); if (rc) return rc;
            if (n > 0) {
                rc = run_layer(c, (int)l, cur, n, ih, iw, L.raw, false); if (rc) return rc;
                CU(maxpool2x2(L.raw, n, ih, iw, L.cs_out, dst, c->stream));
                c->launches++;
            }
        } else if (n > 0) { rc = run_layer(c, (int)l, cur, n, ih, iw, dst, true, in_split, L.xsplit); if (rc) return rc; }
        tick(c);
        cur = dst; h = oh; w = ow;
    }
    c->last_n = n;
    if (d_pred) *d_pred = c->layers.back().view;
    if (gh) *gh = c->layers.back().oh;
    if (gw) *gw = c->layers.back().ow;
    return 0;
}

int yolo_b200_backbone(yolo_b200_ctx *c, const int8_t *d_nhwc4, int n, int h, int w, const int8_t **d_pred, int *gh, int *gw)
{
    int rc = check_ready(c, n, h, w); if (rc) return rc;
    if (!d_nhwc4 && n > 0) return fail(E_ARG, "null input");
    c->ev_used = 0;
    tick(c);
    return backbone_from(c, 0, d_nhwc4, n, h, w, d_pred, gh, gw);
}

// Tracker pass on the GPU (SURVEY 8f rank 3): one forward pass over a float NCHW batch that visits every
// AveragedRangeTracker (slim_yolo_v2.py:9-38) in order.  The activations are exact dyadic rationals y = num * 2^-E, so
// max|a| of each tracker's input comes from integer max/min reductions of the layer numerators: each layer is run twice,
// once to reduce (conv_direct.cu statistics mode) and once, with the exponents then in force, to produce the quantised map the
// next layer sees.
//   TRK_FIRST   fresh trackers: scale = 127 / max|a| (first-call rule, :22-27); retune[l] = largest r with max|y_l| * 2^r < 2^15
//               (the overflow guard of find=True, :222-227; retune_bias_quantize_findbest.py:115-148)
//   TRK_EMA     scale <- scale * (1 - momentum) + (127 / max|a|) * momentum for trackers that have been called before
//               (scale != 0), first-call rule for the others (:25-31): a calibration set larger than one batch
//   TRK_MEASURE nothing changes: reports max|a| per tracker under the tables in force (the `find` assertion, :222-226)
// The exponent a tracker quantises with is floor(log2(scale)) (:33).  All arithmetic on the maxima follows the reference's
// float32 tensor operations.  The context's tables are changed only if the whole pass succeeds.
enum { TRK_FIRST = 0, TRK_EMA = 1, TRK_MEASURE = 2 };

static int reprogram_all(yolo_b200_ctx *c)
{
    build_rgb444_lut(c->prm.scale_a[0], c->lut_host);
    CU(upload(c, c->lut_dev, c->lut_host, sizeof c->lut_host));
    c->lut8_saturates = build_u8_lut(c->prm.scale_a[0], c->lut8_host);
    CU(upload(c, c->lut8_dev, c->lut8_host, sizeof c->lut8_host));
    for (size_t l = 0; l < c->layers.size(); ++l) { int rc = derive_layer(c, (int)l); if (rc) return rc; }
    return 0;
}

static int tracker_pass_inner(yolo_b200_ctx *c, const float *d_nchw, int n, int h, int w, int mode, float momentum,
                              float *scales /*[L+1], in/out, may be NULL*/, double *max_abs /*[L+1], may be NULL*/)
{
    yolo_b200_params &p = c->prm;
    int hs[2], rc;
    if (c->graph) return fail(E_UNSUPPORTED, "the tracker pass covers plain chains of 3x3 layers (slim_yolo_v2); calibrate yolo_v2 with the exporter");
    auto new_scale = [&](int t, float m32) -> float {                 // tracker t sees max|a| = m32 (float32, as the tensor op yields)
        const float fresh = 127.0f / m32;
        if (mode == TRK_FIRST || !scales || scales[t] == 0.f) return fresh;
        return scales[t] * (1.0f - momentum) + fresh * momentum;      // self.scale.mul_(1 - m).add_(scale * m), float32
    };
    // input tracker
    CU(cudaMemsetAsync(c->stats_dev, 0, 2 * sizeof(int), c->stream));
    CU(absmax_f32(d_nchw, (size_t)n * 3 * h * w, reinterpret_cast<unsigned *>(c->stats_dev), c->stream));
    c->launches++;
    CU(cudaMemcpyAsync(hs, c->stats_dev, sizeof hs, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    float m32; memcpy(&m32, &hs[0], 4);
    if (!(m32 > 0.f) || !isfinite(m32)) return fail(E_ARG, "tracker pass: input is all zero or not finite");
    if (max_abs) max_abs[0] = (double)m32;
    if (mode != TRK_MEASURE) {
        const float sc = new_scale(0, m32);
        if (scales) scales[0] = sc;
        p.scale_a[0] = (int)floorf(log2f(sc));
        build_rgb444_lut(p.scale_a[0], c->lut_host);
        CU(upload(c, c->lut_dev, c->lut_host, sizeof c->lut_host));
        c->lut8_saturates = build_u8_lut(p.scale_a[0], c->lut8_host);
        CU(upload(c, c->lut8_dev, c->lut8_host, sizeof c->lut8_host));
    }
    rc = ensure((void **)&c->in_q, &c->in_q_cap, (size_t)n * h * w * 4); if (rc) return rc;
    rc = yolo_b200_quantize_f32(c, d_nchw, n, h, w, c->in_q); if (rc) return rc;
    const int8_t *cur = c->in_q;
    for (size_t l = 0; l < c->layers.size(); ++l) {
        LayerDev &L = c->layers[l];
        const yolo_b200_layer &Lp = p.layers[l];
        if (Lp.pool && (h < 2 || w < 2)) return fail(E_ARG, "input too small: layer %zu pools a %dx%d map", l, h, w);
        // statistics pass: numerator at scale E = max(sa_i + sw, sb), biases shifted accordingly (|acc << la| < 2^28 and
        // |b << lb| <= 2^30 by the limits below: the int32 numerator cannot wrap)
        const int ea = p.scale_a[l] + p.scale_w[l], E = ea > p.scale_b[l] ? ea : p.scale_b[l];
        const int la = E - ea, lb = E - p.scale_b[l];
        if (la > 6 || lb > 23 || la < 0) return fail(E_UNSUPPORTED, "layer %zu: exponents out of range in the tracker pass (la %d lb %d)", l, la, lb);
        std::vector<int> bp(L.cout_pad, 0);
        for (int o = 0; o < L.cout; ++o) bp[o] = (int)L.bias_host[o] * (1 << lb);
        CU(upload(c, L.bias_sh, bp.data(), bp.size() * sizeof(int)));
        const int init[2] = { INT32_MIN, INT32_MAX };
        CU(cudaMemcpyAsync(c->stats_dev, init, sizeof init, cudaMemcpyHostToDevice, c->stream));
        ConvArgs a;
        fill_args(c, (int)l, cur, n, h, w, nullptr, a);
        a.q.la = la; a.stats = c->stats_dev;
        CU(conv3x3_direct(a, c->stream));
        c->launches++;
        CU(cudaMemcpyAsync(hs, c->stats_dev, sizeof hs, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        const double pos = hs[0] > 0 ? (double)hs[0] : 0.0;
        double neg = hs[1] < 0 ? -(double)hs[1] : 0.0;
        if (Lp.activ) neg *= 0.125;                                    // leaky-ReLU before the tracker (slim_yolo_v2.py:220-229)
        const double md = ldexp(pos > neg ? pos : neg, -E);            // max |y|, exact (|numerator| < 2^31, a power-of-two scale)
        if (!(md > 0.0)) return fail(E_ARG, "layer %zu produces only zeros on this batch", l);
        if (max_abs) max_abs[l + 1] = md;
        if (mode != TRK_MEASURE) {
            if (mode == TRK_FIRST || !scales || scales[l + 1] == 0.f) {   // the accumulator scale is tuned with the trackers' first call
                int r = (int)floor(log2(32768.0 / md));
                while (md * ldexp(1.0, r) >= 32768.0) --r;
                p.retune[l] = r;
            }
            const float sc = new_scale((int)l + 1, (float)md);
            if (scales) scales[l + 1] = sc;
            p.scale_a[l + 1] = (int)floorf(log2f(sc));
        }
        rc = derive_layer(c, (int)l); if (rc) return rc;              // (also restores the epilogue's biases after the statistics pass)
        // the layer itself, with the exponents in force
        const int oh = Lp.pool ? h / 2 : h, ow = Lp.pool ? w / 2 : w;
        rc = ensure((void **)&L.out, &L.out_cap, (size_t)n * oh * ow * L.cs_out); if (rc) return rc;
        L.oh = oh; L.ow = ow; L.view = L.out; L.xsplit = false;
        rc = run_layer(c, (int)l, cur, n, h, w, L.out); if (rc) return rc;
        cur = L.out; h = oh; w = ow;
    }
    c->last_n = n;
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

static int tracker_pass(yolo_b200_ctx *c, const float *d_nchw, int n, int h, int w, int mode, float momentum, float *scales, double *max_abs)
{
    int rc = check_ready(c, n, h, w); if (rc) return rc;
    if (!d_nchw || n < 1) return fail(E_ARG, "the tracker pass needs at least one frame");
    if (((size_t)h * w) % 4) return fail(E_UNSUPPORTED, "h*w must be a multiple of 4");
    if (mode == TRK_EMA && !(momentum >= 0.f && momentum <= 1.f)) return fail(E_ARG, "momentum %g", (double)momentum);
    const yolo_b200_params saved = c->prm;
    std::vector<float> sc_saved;
    if (scales) sc_saved.assign(scales, scales + c->prm.num_layers + 1);
    rc = tracker_pass_inner(c, d_nchw, n, h, w, mode, momentum, scales, max_abs);
    if (rc) {
        // leave the context exactly as it was: tables, look-up tables and every layer's epilogue programme
        char msg[sizeof g_err];
        memcpy(msg, g_err, sizeof msg);
        c->prm = saved;
        if (scales) memcpy(scales, sc_saved.data(), sc_saved.size() * sizeof(float));
        if (reprogram_all(c)) c->loaded = false;
        memcpy(g_err, msg, sizeof msg);
    }
    return rc;
}

int yolo_b200_calibrate_f32(yolo_b200_ctx *c, const float *d_nchw, int n, int h, int w, int32_t *scale_a_out, int32_t *retune_out)
{
    int rc = tracker_pass(c, d_nchw, n, h, w, TRK_FIRST, 0.f, nullptr, nullptr); if (rc) return rc;
    const yolo_b200_params &p = c->prm;
    if (scale_a_out) for (int l = 0; l <= p.num_layers; ++l) scale_a_out[l] = p.scale_a[l];
    if (retune_out) for (int l = 0; l < p.num_layers; ++l) retune_out[l] = p.retune[l];
    return 0;
}

int yolo_b200_update_trackers_f32(yolo_b200_ctx *c, const float *d_nchw, int n, int h, int w, float momentum,
                                  float *tracker_scale, int32_t *scale_a_out, int32_t *retune_out)
{
    if (!tracker_scale) return fail(E_ARG, "null tracker_scale");
    int rc = tracker_pass(c, d_nchw, n, h, w, TRK_EMA, momentum, tracker_scale, nullptr); if (rc) return rc;
    const yolo_b200_params &p = c->prm;
    if (scale_a_out) for (int l = 0; l <= p.num_layers; ++l) scale_a_out[l] = p.scale_a[l];
    if (retune_out) for (int l = 0; l < p.num_layers; ++l) retune_out[l] = p.retune[l];
    return 0;
}

int yolo_b200_measure_f32(yolo_b200_ctx *c, const float *d_nchw, int n, int h, int w, double *max_abs)
{
    if (!max_abs) return fail(E_ARG, "null max_abs");
    return tracker_pass(c, d_nchw, n, h, w, TRK_MEASURE, 0.f, nullptr, max_abs);
}

int yolo_b200_get_layer_output(yolo_b200_ctx *c, int layer, int8_t *host_out, size_t bytes)
{
    if (!c || !host_out) return fail(E_ARG, "null argument");
    if (layer < 0 || layer >= (int)c->layers.size()) return fail(E_ARG, "layer %d out of range", layer);
    LayerDev &L = c->layers[layer];
    size_t have = (size_t)c->last_n * L.oh * L.ow * L.cs_out;
    if (bytes != have) return fail(E_ARG, "layer %d output is %zu bytes, caller passed %zu", layer, have, bytes);
    CU(cudaSetDevice(c->device));
    CU(cudaMemcpyAsync(host_out, L.view ? L.view : L.out, bytes, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (L.xsplit) {
        // the chain kept this map with its rows split by x parity ([even pixels][odd pixels]): hand out plain NHWC
        const size_t px = (size_t)L.cs_out, row = (size_t)L.ow * px, half = (size_t)(L.ow / 2);
        std::vector<int8_t> tmp(row);
        for (size_t r = 0; r < (size_t)c->last_n * L.oh; ++r) {
            int8_t *p = host_out + r * row;
            memcpy(tmp.data(), p, row);
            for (size_t x = 0; x < (size_t)L.ow; ++x) memcpy(p + x * px, tmp.data() + ((x & 1) * half + (x >> 1)) * px, px);
        }
    }
    return 0;
}

// scratch of the head (scores, classes, boxes of every anchor) for `frames` frames
static int ensure_head(yolo_b200_ctx *c, size_t frames, size_t N)
{
    if (c->head_cap >= frames * N) return 0;
    cudaFree(c->h_scores); cudaFree(c->h_cls); cudaFree(c->h_boxes);
    c->h_scores = nullptr; c->h_cls = nullptr; c->h_boxes = nullptr; c->head_cap = 0;
    CU(cudaMalloc(&c->h_scores, frames * N * sizeof(float)));
    CU(cudaMalloc(&c->h_cls, frames * N * sizeof(int)));
    CU(cudaMalloc(&c->h_boxes, frames * N * sizeof(float4)));
    c->head_cap = frames * N;
    return 0;
}

// decode + NMS of n frames on stream st; the frames use the scratch slots [slot0, slot0 + n) (ensure_head first)
static int detect_on(yolo_b200_ctx *c, cudaStream_t st, size_t slot0, const int8_t *d_pred, int n, int gh, int gw, int in_h, int in_w,
                     yolo_b200_det *d_dets, int32_t *d_counts)
{
    const yolo_b200_params &p = c->prm;
    const size_t N = (size_t)gh * gw * p.num_anchors;
    HeadArgs a;
    a.pred = d_pred; a.n = n; a.gh = gh; a.gw = gw; a.cs = yolo_b200_cstride(p.num_anchors * (5 + p.num_classes));
    a.A = p.num_anchors; a.C = p.num_classes; a.sa_pred = p.scale_a[p.num_layers];
    for (int i = 0; i < YOLO_B200_MAX_ANCHORS; ++i) { a.anchors[i][0] = p.anchors[i][0]; a.anchors[i][1] = p.anchors[i][1]; }
    a.stride = p.stride; a.in_h = in_h; a.in_w = in_w; a.conf_thresh = p.conf_thresh; a.nms_thresh = p.nms_thresh;
    a.head_mode = p.head_mode; a.max_det = p.max_det;
    a.scores = c->h_scores + slot0 * N; a.cls = c->h_cls + slot0 * N; a.boxes = c->h_boxes + slot0 * N; a.dets = d_dets; a.counts = d_counts;
    a.fused_decode = head_nms_fuses_decode(a) ? 1 : 0;
    if (!a.fused_decode) { CU(head_decode(a, st)); c->launches++; }
    CU(head_nms(a, st));
    c->launches++;
    return 0;
}

int yolo_b200_detect(yolo_b200_ctx *c, const int8_t *d_pred, int n, int gh, int gw, int in_h, int in_w,
                     yolo_b200_det *d_dets, int32_t *d_counts)
{
    int rc = check_ready(c, n, gh, gw); if (rc) return rc;
    if (n == 0) return 0;
    if (!d_pred || !d_dets || !d_counts) return fail(E_ARG, "null buffer");
    const size_t N = (size_t)gh * gw * c->prm.num_anchors;
    if (N > (size_t)HEAD_MAX_CAND) return fail(E_UNSUPPORTED, "grid %dx%d x %d anchors exceeds %d candidates per frame", gh, gw, c->prm.num_anchors, HEAD_MAX_CAND);
    rc = ensure_head(c, (size_t)n, N); if (rc) return rc;
    rc = detect_on(c, c->stream, 0, d_pred, n, gh, gw, in_h, in_w, d_dets, d_counts); if (rc) return rc;
    tick(c);
    return 0;
}

int yolo_b200_forward_int8_dev(yolo_b200_ctx *c, const int8_t *d_nhwc4, int n, int h, int w, yolo_b200_det *d_dets, int32_t *d_counts)
{
    const int8_t *pred; int gh, gw;
    int rc = yolo_b200_backbone(c, d_nhwc4, n, h, w, &pred, &gh, &gw); if (rc) return rc;
    return yolo_b200_detect(c, pred, n, gh, gw, h, w, d_dets, d_counts);
}

// Camera / image front ends fused into the first layer (auto back end): the quantised frame never exists in HBM.
// IN_RGB444 (camera_to_inpBuf + pixel_norm_quantize, yolo_forward.c:57-123), IN_BGR (BaseTransform + tracker).
static int fused_front_features(yolo_b200_ctx *c, InKind kind, const void *d_src, int n, int h, int w, int8_t *last_out,
                                const int8_t **pred, int *gh, int *gw, bool *done)
{
    *done = false;
    LayerDev &L0 = c->layers[0];
    ConvArgs a0;
    fill_args(c, 0, nullptr, n, h, w, nullptr, a0);
    if (!(n > 0 && c->conv_backend == 0 && c->layers.size() > 1 && conv3x3_first_supported(a0) && conv3x3_first_src_ok(kind, d_src) && !(L0.q.pool && (h < 2 || w < 2)))) return 0;
    if (kind == IN_RGB444 && (((uintptr_t)d_src) & 1)) return 0;
    if (kind == IN_BGR && c->lut8_saturates) return 0;              // saturated inputs must be counted: the stand-alone quantiser does
    const int oh = L0.q.pool ? h / 2 : h, ow = L0.q.pool ? w / 2 : w;
    int rc = ensure((void **)&L0.out, &L0.out_cap, (size_t)n * oh * ow * L0.cs_out); if (rc) return rc;
    L0.oh = oh; L0.ow = ow; L0.rh = h; L0.rw = w; L0.view = L0.out;
    a0.out = L0.out;
    L0.xsplit = want_xsplit(c, 0, d_src, n, oh, ow);
    a0.out_xsplit = L0.xsplit;
    c->ev_used = 0;
    tick(c);
    CU(conv3x3_first(a0, c->stream, kind, d_src, kind == IN_RGB444 ? (const void *)c->lut_dev : (const void *)c->lut8_dev));
    c->launches += conv3x3_fs_supported(a0, kind, d_src) ? 1 : L0.cs_out / 16;
    tick(c);
    rc = backbone_from(c, 1, L0.out, n, oh, ow, pred, gh, gw, last_out); if (rc) return rc;
    *done = true;
    return 0;
}

// Front end + all convolution layers for one of the four input kinds.
static int features_dev(yolo_b200_ctx *c, InKind kind, const void *d_src, int n, int h, int w, int8_t *last_out,
                        const int8_t **pred, int *gh, int *gw)
{
    int rc = check_ready(c, n, h, w); if (rc) return rc;
    if (!d_src && n > 0) return fail(E_ARG, "null input");
    if (kind == IN_RGB444 || kind == IN_BGR) {
        bool done;
        rc = fused_front_features(c, kind, d_src, n, h, w, last_out, pred, gh, gw, &done);
        if (rc || done) return rc;
    }
    const int8_t *x8 = (const int8_t *)d_src;
    if (kind != IN_INT8) {
        rc = ensure((void **)&c->in_q, &c->in_q_cap, (size_t)(n > 0 ? n : 1) * h * w * 4); if (rc) return rc;
        if (kind == IN_RGB444) rc = yolo_b200_quantize_rgb444(c, (const uint16_t *)d_src, n, h, w, c->in_q);
        else if (kind == IN_BGR) rc = yolo_b200_quantize_u8bgr(c, (const uint8_t *)d_src, n, h, w, c->in_q);
        else rc = yolo_b200_quantize_f32(c, (const float *)d_src, n, h, w, c->in_q);
        if (rc) return rc;
        x8 = c->in_q;
    }
    c->ev_used = 0;
    tick(c);
    return backbone_from(c, 0, x8, n, h, w, pred, gh, gw, last_out);
}

static int forward_dev(yolo_b200_ctx *c, InKind kind, const void *d_src, int n, int h, int w, yolo_b200_det *d_dets, int32_t *d_counts)
{
    const int8_t *pred; int gh, gw;
    int rc = features_dev(c, kind, d_src, n, h, w, nullptr, &pred, &gh, &gw); if (rc) return rc;
    return yolo_b200_detect(c, pred, n, gh, gw, h, w, d_dets, d_counts);
}

// The device forward of the resize front ends: plan, resize into the context's buffer, forward_dev
static int forward_resize_dev(yolo_b200_ctx *c, int fmt, const uint8_t *d_src, int n, const int32_t *src_hw, int stride, int h, int w,
                              yolo_b200_det *d_dets, int32_t *d_counts, const yolo_b200_frames *layout = nullptr)
{
    int rc = check_ready(c, n, h, w); if (rc) return rc;
    SourcePlan p;
    rc = plan_sources(fmt, n, src_hw, stride, h, w, true, p, layout); if (rc) return rc;
    if (n == 0) return 0;
    if (!d_src || !d_dets || !d_counts) return fail(E_ARG, "null buffer");
    if (p.mode != RESIZE_NONE) {
        rc = ensure((void **)&c->rs_out, &c->rs_out_cap, (size_t)n * h * w * 3); if (rc) return rc;
        rc = resize_dev(c, p, d_src, c->rs_out); if (rc) return rc;
        d_src = c->rs_out;
    }
    return forward_dev(c, IN_BGR, d_src, n, h, w, d_dets, d_counts);
}

int yolo_b200_forward_rgb444_dev(yolo_b200_ctx *c, const uint16_t *d_frames, int n, int h, int w, yolo_b200_det *d_dets, int32_t *d_counts)
{ return forward_dev(c, IN_RGB444, d_frames, n, h, w, d_dets, d_counts); }

int yolo_b200_forward_u8bgr_dev(yolo_b200_ctx *c, const uint8_t *d_bgr, int n, int h, int w, yolo_b200_det *d_dets, int32_t *d_counts)
{ return forward_dev(c, IN_BGR, d_bgr, n, h, w, d_dets, d_counts); }

int yolo_b200_forward_u8bgr_resize_dev(yolo_b200_ctx *c, const uint8_t *d_bgr, int n, int sh, int sw, int h, int w,
                                       yolo_b200_det *d_dets, int32_t *d_counts)
{
    const int32_t hw[2] = { sh, sw };
    return forward_resize_dev(c, RS_BGR, d_bgr, n, hw, 0, h, w, d_dets, d_counts);
}

int yolo_b200_forward_u8bgr_ragged_dev(yolo_b200_ctx *c, const uint8_t *d_bgr, int n, const int32_t *src_hw, int h, int w,
                                       yolo_b200_det *d_dets, int32_t *d_counts)
{ return forward_resize_dev(c, RS_BGR, d_bgr, n, src_hw, 1, h, w, d_dets, d_counts); }

int yolo_b200_forward_yuv_dev(yolo_b200_ctx *c, const uint8_t *d_frames, int format, int n, int sh, int sw, int h, int w,
                              yolo_b200_det *d_dets, int32_t *d_counts)
{
    const int32_t hw[2] = { sh, sw };
    return forward_resize_dev(c, yuv_format(format), d_frames, n, hw, 0, h, w, d_dets, d_counts);
}

int yolo_b200_forward_bayer_dev(yolo_b200_ctx *c, const uint8_t *d_frames, int pattern, int n, int sh, int sw, int h, int w,
                                yolo_b200_det *d_dets, int32_t *d_counts)
{
    const int32_t hw[2] = { sh, sw };
    return forward_resize_dev(c, bayer_format(pattern), d_frames, n, hw, 0, h, w, d_dets, d_counts);
}

int yolo_b200_forward_pix_dev(yolo_b200_ctx *c, const uint8_t *d_frames, int format, int n, int sh, int sw, int h, int w,
                              yolo_b200_det *d_dets, int32_t *d_counts)
{
    const int32_t hw[2] = { sh, sw };
    return forward_resize_dev(c, pix_format(format), d_frames, n, hw, 0, h, w, d_dets, d_counts);
}

int yolo_b200_forward_frames_dev(yolo_b200_ctx *c, const uint8_t *d_frames, const yolo_b200_frames *d, int n, int h, int w,
                                 yolo_b200_det *d_dets, int32_t *d_counts)
{
    YB_FRAMES(d);
    return forward_resize_dev(c, fmt, d_frames, n, hw, 0, h, w, d_dets, d_counts, d);
}

int yolo_b200_forward_f32_dev(yolo_b200_ctx *c, const float *d_nchw, int n, int h, int w, yolo_b200_det *d_dets, int32_t *d_counts)
{ return forward_dev(c, IN_F32, d_nchw, n, h, w, d_dets, d_counts); }

int yolo_b200_sync(yolo_b200_ctx *c)
{
    if (!c) return fail(E_ARG, "null ctx");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

// host-buffer variants: H2D of the frames, forward, D2H of detections + counts.  The frames travel and are convolved chunk
// by chunk over two streams (the copy of chunk k+1 overlaps the convolution layers of chunk k; frames are independent, so
// chunking changes no result); every chunk's prediction map lands in one batch-wide buffer and decode + NMS then run once
// over the whole batch (a per-chunk NMS launch cannot fill the GPU: it is one CTA per frame).  Only the filled part of the
// detection lists is copied back.
// The plan p says where the host frames are and how they are resized to the network size on the GPU, chunk by chunk,
// between the copy and the first layer: chunk k's copy is the byte range [at(f0), at(f0 + nk)) of the host buffer, and
// enqueue_resize makes its landed frames network input.  A ragged plan's descriptors and tables go into the slot's own
// buffers, uploaded on the copy stream (the slot's previous call has completed, so nothing queued still reads them).
// host_enqueue queues the whole call (copies in, layers, decode + NMS, copy of the counts) on the context's streams and
// returns; host_complete waits for the counts, copies the filled part of the lists back and waits for that copy.
static int host_enqueue(yolo_b200_ctx *c, int si, const void *host_in, const SourcePlan &p, yolo_b200_det *dets, int32_t *counts)
{
    HostSlot &S = c->slots[si];
    S.ngroups = 0; S.dets = dets; S.counts = counts;
    const int n = p.n, h = p.dh, w = p.dw;
    const bool resize = p.mode != RESIZE_NONE;
    const size_t net_frame_bytes = resize ? (size_t)h * w * 3 : p.frame_bytes;
    int rc = ensure(&S.stage_in, &S.stage_in_cap, (size_t)n * net_frame_bytes); if (rc) return rc;
    if (resize) { rc = ensure(&S.rs_src, &S.rs_src_cap, p.end(0, n) - p.first); if (rc) return rc; }
    const size_t md = (size_t)c->prm.max_det;
    rc = ensure((void **)&S.d_dets, &S.dets_cap, (size_t)n * md * sizeof(yolo_b200_det)); if (rc) return rc;
    rc = ensure((void **)&S.d_counts, &S.counts_cap, (size_t)n * sizeof(int32_t)); if (rc) return rc;
    // prediction map of the whole batch
    int gh = h, gw = w;
    for (auto &L : c->layers) {
        if (L.q.pool && (gh < 2 || gw < 2)) return fail(E_ARG, "input too small for the pooling layers");
        if (L.q.pool) { gh /= 2; gw /= 2; }
    }
    const size_t pred_frame = (size_t)gh * gw * c->layers.back().cs_out;
    rc = ensure((void **)&S.pred_all, &S.pred_all_cap, (size_t)n * pred_frame); if (rc) return rc;
    const int chunk = c->host_chunk > 0 ? c->host_chunk : n;
    std::vector<int> cf0, cnk;                                   // first frame / frames of each chunk
    if (const char *sched = getenv("YOLO_B200_CHUNKS")) {        // experiment hook: explicit chunk sizes, the last one repeats
        int f = 0, last = chunk;
        while (f < n) {
            if (sched && *sched) { last = atoi(sched); sched = strchr(sched, ','); if (sched) ++sched; }
            if (last < 1) last = chunk;
            const int nk = (n - f) < last ? (n - f) : last;
            cf0.push_back(f); cnk.push_back(nk); f += nk;
        }
    } else {
        for (int f = 0; f < n; f += chunk) { cf0.push_back(f); cnk.push_back((n - f) < chunk ? (n - f) : chunk); }
    }
    const int nchunks = (int)cf0.size();
    const size_t N = (size_t)gh * gw * c->prm.num_anchors;
    if (N > (size_t)HEAD_MAX_CAND) return fail(E_UNSUPPORTED, "grid %dx%d x %d anchors exceeds %d candidates per frame", gh, gw, c->prm.num_anchors, HEAD_MAX_CAND);
    rc = ensure_head(c, (size_t)n, N); if (rc) return rc;
    if (S.counts_pinned_cap < (size_t)n) {
        if (S.counts_pinned) cudaFreeHost(S.counts_pinned);
        S.counts_pinned = nullptr; S.counts_pinned_cap = 0;
        CU(cudaHostAlloc((void **)&S.counts_pinned, (size_t)n * sizeof(int32_t), cudaHostAllocDefault));
        S.counts_pinned_cap = (size_t)n;
    }
    if (!c->s_in) {
        CU(cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&c->s_head, cudaStreamNonBlocking));
    }
    if (!S.ev_out) CU(cudaEventCreateWithFlags(&S.ev_out, cudaEventDisableTiming));
    auto grow = [](std::vector<cudaEvent_t> &v, int want) -> cudaError_t {
        while ((int)v.size() < want) {
            cudaEvent_t e1;
            cudaError_t e = cudaEventCreateWithFlags(&e1, cudaEventDisableTiming);
            if (e != cudaSuccess) return e;
            v.push_back(e1);
        }
        return cudaSuccess;
    };
    CU(grow(S.ev_in, nchunks)); CU(grow(S.ev_done, nchunks)); CU(grow(S.ev_cnt, nchunks));
    auto drain = [&]() { cudaStreamSynchronize(c->s_in); cudaStreamSynchronize(c->stream); cudaStreamSynchronize(c->s_head); cudaStreamSynchronize(c->s_out); };
    HostTrace &tr = S.tr;
    tr.ev.clear();
    tr.on = getenv("YOLO_B200_TRACE_HOST") != nullptr;
    if (tr.on) { cudaEventCreate(&tr.t0); cudaEventRecord(tr.t0, c->s_in); }
    const ResizeTables *tabs = nullptr;
    rc = resize_tables(c, p, S.tabs, c->s_in, &tabs); if (rc) return rc;
    // The slot's buffers are its own: nothing queued earlier reads or writes them once the slot's previous call has been
    // completed, so the copies of this call do NOT wait for the context stream (the layers of the previous call may still
    // be running there: that overlap is the point of the second slot).
    // Three stages, all queued up front: chunk k's frames are copied in on s_in, its convolution layers run on the
    // context stream, decode + NMS and the copy of the counts on s_head.  The head runs twice: once for all chunks but the
    // last, as soon as the second-to-last chunk's layers are done (it then overlaps the last chunk's copy, which the GPU
    // would otherwise wait for), and once for the last chunk.  (A head per chunk was measured slower: the NMS CTAs hold
    // shared memory the persistent convolution CTAs of the next chunk need, so the two serialise.)
    int head_f0 = 0;
    size_t landed = 0;                                           // host bytes below this are already copied (or queued)
    for (int k = 0; k < nchunks; ++k) {
        const int f0 = cf0[k], nk = cnk[k];
        char *stage = (char *)S.stage_in + (size_t)f0 * net_frame_bytes;
        // host byte p.begin(0) + b lands at rs_src + b: a pitched chunk is its span, padding included.  Where frames overlap
        // (stride below a frame's span) the chunk copies only what earlier chunks have not, so no copy writes bytes an
        // earlier chunk's resize reads; those landed before this chunk's copy (s_in is in order), which its resize waits for.
        char *land = resize ? (char *)S.rs_src + p.at(f0) : stage;
        const size_t from = std::max(p.begin(f0), landed), to = p.end(f0, nk);
        if (to > from)
            CU(cudaMemcpyAsync(land + (from - p.begin(f0)), (const char *)host_in + from, to - from, cudaMemcpyHostToDevice, c->s_in));
        landed = std::max(landed, to);
        CU(cudaEventRecord(S.ev_in[k], c->s_in));
        tr.mark("h2d done", k, c->s_in);
        CU(cudaStreamWaitEvent(c->stream, S.ev_in[k], 0));
        if (resize) {
            cudaError_t e = enqueue_resize(c, p, *tabs, (const uint8_t *)S.rs_src, f0, nk, (uint8_t *)stage);
            if (e != cudaSuccess) { drain(); return fail(E_CUDA, "resize: %s", cudaGetErrorString(e)); }
        }
        const int8_t *pred; int g1, g2;
        rc = features_dev(c, p.kind, stage, nk, h, w, S.pred_all + (size_t)f0 * pred_frame, &pred, &g1, &g2);
        if (rc) { drain(); return rc; }
        tr.mark("layers done", k, c->stream);
        if (k == nchunks - 2 || k == nchunks - 1) {
            const int hn = f0 + nk - head_f0;                                  // frames [head_f0, f0 + nk)
            CU(cudaEventRecord(S.ev_done[S.ngroups], c->stream));
            CU(cudaStreamWaitEvent(c->s_head, S.ev_done[S.ngroups], 0));
            rc = detect_on(c, c->s_head, (size_t)head_f0, S.pred_all + (size_t)head_f0 * pred_frame, hn, gh, gw, h, w,
                           S.d_dets + (size_t)head_f0 * md, S.d_counts + head_f0);
            if (rc) { drain(); return rc; }
            CU(cudaMemcpyAsync(S.counts_pinned + head_f0, S.d_counts + head_f0, (size_t)hn * sizeof(int32_t), cudaMemcpyDeviceToHost, c->s_head));
            CU(cudaEventRecord(S.ev_cnt[S.ngroups], c->s_head));
            tr.mark("head+counts done", S.ngroups, c->s_head);
            S.grp_f0[S.ngroups] = head_f0; S.grp_n[S.ngroups] = hn; ++S.ngroups;
            head_f0 = f0 + nk;
        }
    }
    S.busy = true;
    return 0;
}

static int host_complete(yolo_b200_ctx *c, int si)
{
    HostSlot &S = c->slots[si];
    if (!S.busy) return fail(E_STATE, "nothing in flight on ticket %d", si);
    S.busy = false;
    auto drain = [&]() { cudaStreamSynchronize(c->s_in); cudaStreamSynchronize(c->stream); cudaStreamSynchronize(c->s_head); cudaStreamSynchronize(c->s_out); };
    const size_t md = (size_t)c->prm.max_det;
    // detections: per head launch, one strided copy as wide as its largest count, as soon as its counts are here
    for (int k = 0; k < S.ngroups; ++k) {
        const int f0 = S.grp_f0[k], nk = S.grp_n[k];
        cudaError_t e = cudaEventSynchronize(S.ev_cnt[k]);
        if (e != cudaSuccess) { drain(); return fail(E_CUDA, "%s", cudaGetErrorString(e)); }
        int maxc = 0;
        for (int i = 0; i < nk; ++i) { S.counts[f0 + i] = S.counts_pinned[f0 + i]; maxc = S.counts[f0 + i] > maxc ? S.counts[f0 + i] : maxc; }
        if (maxc > (int)md) maxc = (int)md;
        if (maxc > 0)
            CU(cudaMemcpy2DAsync(S.dets + (size_t)f0 * md, md * sizeof(yolo_b200_det), S.d_dets + (size_t)f0 * md, md * sizeof(yolo_b200_det),
                                 (size_t)maxc * sizeof(yolo_b200_det), (size_t)nk, cudaMemcpyDeviceToHost, c->s_out));
        S.tr.mark("dets d2h done", k, c->s_out);
    }
    CU(cudaEventRecord(S.ev_out, c->s_out));
    CU(cudaEventSynchronize(S.ev_out));       // the lists are in the caller's buffers (everything the call queued has finished before them)
    S.tr.dump();
    S.tr.on = false;
    return 0;
}

static int host_free_slot(yolo_b200_ctx *c)
{
    for (int i = 0; i < YB_HOST_SLOTS; ++i) if (!c->slots[i].busy) return i;
    return -1;
}

// The host-buffer calls, frames at host_in as plan p says.  Blocking (submit == false): submit + wait on any free slot,
// n == 0 is a no-op.  Asynchronous (submit == true, n >= 1): returns a ticket (>= 0) once the call is queued; the caller's
// buffers belong to the library until yolo_b200_wait(ticket) returns.
static int host_call(yolo_b200_ctx *c, bool submit, const void *host_in, const SourcePlan &p, yolo_b200_det *dets, int32_t *counts)
{
    int rc = check_ready(c, p.n, p.dh, p.dw); if (rc) return rc;
    if (submit && p.n < 1) return fail(E_ARG, "submit needs n >= 1");
    if (p.n == 0) return 0;
    if (!host_in || !dets || !counts) return fail(E_ARG, "null buffer");
    const int si = host_free_slot(c);
    if (si < 0) return fail(E_STATE, "%d submissions in flight: call yolo_b200_wait first", YB_HOST_SLOTS);
    rc = host_enqueue(c, si, host_in, p, dets, counts); if (rc) return rc;
    return submit ? si : host_complete(c, si);
}

// host calls of the resize front ends (sizes as plan_sources reads them)
static int host_resize(yolo_b200_ctx *c, bool submit, int fmt, const void *host_in, int n, const int32_t *src_hw, int stride, int h, int w,
                       yolo_b200_det *dets, int32_t *counts, const yolo_b200_frames *layout = nullptr)
{
    SourcePlan p;
    int rc = plan_sources(fmt, n, src_hw, stride, h, w, true, p, layout); if (rc) return rc;
    return host_call(c, submit, host_in, p, dets, counts);
}

int yolo_b200_submit_rgb444(yolo_b200_ctx *c, const uint16_t *frames, int n, int h, int w, yolo_b200_det *dets, int32_t *counts)
{ return host_call(c, true, frames, net_plan(IN_RGB444, n, h, w), dets, counts); }
int yolo_b200_submit_u8bgr(yolo_b200_ctx *c, const uint8_t *bgr, int n, int h, int w, yolo_b200_det *dets, int32_t *counts)
{ return host_call(c, true, bgr, net_plan(IN_BGR, n, h, w), dets, counts); }
int yolo_b200_submit_u8bgr_ragged(yolo_b200_ctx *c, const uint8_t *bgr, int n, const int32_t *src_hw, int h, int w,
                                  yolo_b200_det *dets, int32_t *counts)
{ return host_resize(c, true, RS_BGR, bgr, n, src_hw, 1, h, w, dets, counts); }
int yolo_b200_wait(yolo_b200_ctx *c, int ticket)
{
    if (!c) return fail(E_ARG, "null ctx");
    if (ticket < 0 || ticket >= YB_HOST_SLOTS) return fail(E_ARG, "ticket %d", ticket);
    CU(cudaSetDevice(c->device));
    return host_complete(c, ticket);
}

int yolo_b200_forward_rgb444(yolo_b200_ctx *c, const uint16_t *frames, int n, int h, int w, yolo_b200_det *dets, int32_t *counts)
{ return host_call(c, false, frames, net_plan(IN_RGB444, n, h, w), dets, counts); }
int yolo_b200_forward_int8(yolo_b200_ctx *c, const int8_t *nhwc4, int n, int h, int w, yolo_b200_det *dets, int32_t *counts)
{ return host_call(c, false, nhwc4, net_plan(IN_INT8, n, h, w), dets, counts); }
int yolo_b200_forward_u8bgr(yolo_b200_ctx *c, const uint8_t *bgr, int n, int h, int w, yolo_b200_det *dets, int32_t *counts)
{ return host_call(c, false, bgr, net_plan(IN_BGR, n, h, w), dets, counts); }
int yolo_b200_forward_f32(yolo_b200_ctx *c, const float *nchw, int n, int h, int w, yolo_b200_det *dets, int32_t *counts)
{ return host_call(c, false, nchw, net_plan(IN_F32, n, h, w), dets, counts); }
int yolo_b200_forward_u8bgr_resize(yolo_b200_ctx *c, const uint8_t *bgr, int n, int sh, int sw, int h, int w, yolo_b200_det *dets, int32_t *counts)
{
    const int32_t hw[2] = { sh, sw };
    return host_resize(c, false, RS_BGR, bgr, n, hw, 0, h, w, dets, counts);
}
int yolo_b200_forward_u8bgr_ragged(yolo_b200_ctx *c, const uint8_t *bgr, int n, const int32_t *src_hw, int h, int w,
                                   yolo_b200_det *dets, int32_t *counts)
{ return host_resize(c, false, RS_BGR, bgr, n, src_hw, 1, h, w, dets, counts); }
int yolo_b200_forward_yuv(yolo_b200_ctx *c, const uint8_t *frames, int format, int n, int sh, int sw, int h, int w,
                          yolo_b200_det *dets, int32_t *counts)
{
    const int32_t hw[2] = { sh, sw };
    return host_resize(c, false, yuv_format(format), frames, n, hw, 0, h, w, dets, counts);
}
int yolo_b200_submit_yuv(yolo_b200_ctx *c, const uint8_t *frames, int format, int n, int sh, int sw, int h, int w,
                         yolo_b200_det *dets, int32_t *counts)
{
    const int32_t hw[2] = { sh, sw };
    return host_resize(c, true, yuv_format(format), frames, n, hw, 0, h, w, dets, counts);
}
int yolo_b200_forward_bayer(yolo_b200_ctx *c, const uint8_t *frames, int pattern, int n, int sh, int sw, int h, int w,
                            yolo_b200_det *dets, int32_t *counts)
{
    const int32_t hw[2] = { sh, sw };
    return host_resize(c, false, bayer_format(pattern), frames, n, hw, 0, h, w, dets, counts);
}
int yolo_b200_submit_bayer(yolo_b200_ctx *c, const uint8_t *frames, int pattern, int n, int sh, int sw, int h, int w,
                           yolo_b200_det *dets, int32_t *counts)
{
    const int32_t hw[2] = { sh, sw };
    return host_resize(c, true, bayer_format(pattern), frames, n, hw, 0, h, w, dets, counts);
}
int yolo_b200_forward_pix(yolo_b200_ctx *c, const uint8_t *frames, int format, int n, int sh, int sw, int h, int w,
                          yolo_b200_det *dets, int32_t *counts)
{
    const int32_t hw[2] = { sh, sw };
    return host_resize(c, false, pix_format(format), frames, n, hw, 0, h, w, dets, counts);
}
int yolo_b200_submit_pix(yolo_b200_ctx *c, const uint8_t *frames, int format, int n, int sh, int sw, int h, int w,
                         yolo_b200_det *dets, int32_t *counts)
{
    const int32_t hw[2] = { sh, sw };
    return host_resize(c, true, pix_format(format), frames, n, hw, 0, h, w, dets, counts);
}
int yolo_b200_forward_frames(yolo_b200_ctx *c, const uint8_t *frames, const yolo_b200_frames *d, int n, int h, int w,
                             yolo_b200_det *dets, int32_t *counts)
{
    YB_FRAMES(d);
    return host_resize(c, false, fmt, frames, n, hw, 0, h, w, dets, counts, d);
}
int yolo_b200_submit_frames(yolo_b200_ctx *c, const uint8_t *frames, const yolo_b200_frames *d, int n, int h, int w,
                            yolo_b200_det *dets, int32_t *counts)
{
    YB_FRAMES(d);
    return host_resize(c, true, fmt, frames, n, hw, 0, h, w, dets, counts, d);
}
#undef YB_FRAMES

// ---- multi-GPU collection of the detection lists -----------------------------------------------------------------
int yolo_b200_pack_detections(yolo_b200_ctx *c, const yolo_b200_det *d_dets, const int32_t *d_counts, int n,
                              yolo_b200_det *d_packed, int32_t *d_offsets)
{
    if (!c) return fail(E_ARG, "null ctx");
    if (n < 0) return fail(E_ARG, "n %d", n);
    if (n == 0) return 0;
    if (!d_dets || !d_counts || !d_packed || !d_offsets) return fail(E_ARG, "null buffer");
    if (((uintptr_t)d_dets | (uintptr_t)d_packed) & 15) return fail(E_ARG, "detection buffers must be 16-byte aligned");
    CU(cudaSetDevice(c->device));
    CU(pack_detections(d_dets, d_counts, n, c->prm.max_det, d_packed, d_offsets, c->stream));
    c->launches += 2;
    return 0;
}

int yolo_b200_ipc_alloc(yolo_b200_ctx *c, size_t bytes, void **d_ptr, unsigned char handle[64])
{
    if (!c || !d_ptr || !handle || bytes == 0) return fail(E_ARG, "bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CU(cudaSetDevice(c->device));
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return fail(E_NOMEM, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
    cudaIpcMemHandle_t h;
    e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return fail(E_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); }
    memcpy(handle, &h, 64);
    *d_ptr = p;
    return 0;
}

int yolo_b200_ipc_open(yolo_b200_ctx *c, const unsigned char handle[64], void **d_ptr)
{
    if (!c || !d_ptr || !handle) return fail(E_ARG, "bad argument");
    CU(cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CU(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}

int yolo_b200_ipc_close(yolo_b200_ctx *c, void *d_ptr, int opened)
{
    if (!c) return fail(E_ARG, "null ctx");
    if (!d_ptr) return 0;
    CU(cudaSetDevice(c->device));
    if (opened) CU(cudaIpcCloseMemHandle(d_ptr)); else CU(cudaFree(d_ptr));
    return 0;
}

int yolo_b200_copy_async(yolo_b200_ctx *c, void *dst, const void *src, size_t bytes, void *cuda_stream)
{
    if (!c) return fail(E_ARG, "null ctx");
    if (bytes == 0) return 0;
    if (!dst || !src) return fail(E_ARG, "null buffer");
    CU(cudaSetDevice(c->device));
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, cuda_stream ? (cudaStream_t)cuda_stream : c->stream));
    return 0;
}

int yolo_b200_overflow_count(yolo_b200_ctx *c, int64_t *count)
{
    if (!c || !count) return fail(E_ARG, "null argument");
    unsigned v = 0;
    CU(cudaSetDevice(c->device));
    CU(cudaMemcpyAsync(&v, c->ovf_dev, sizeof v, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemsetAsync(c->ovf_dev, 0, sizeof v, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    *count = v;
    return 0;
}

int64_t yolo_b200_launch_count(yolo_b200_ctx *c) { return c ? c->launches : 0; }
int64_t yolo_b200_slow_path_count(yolo_b200_ctx *c) { return c ? c->slow_path_launches : 0; }

int yolo_b200_enable_timing(yolo_b200_ctx *c, int enable)
{
    if (!c) return fail(E_ARG, "null ctx");
    c->timing = enable != 0; c->ev_used = 0;
    return 0;
}

int yolo_b200_layer_times_ms(yolo_b200_ctx *c, float *ms, int capacity)
{
    if (!c || !ms) return fail(E_ARG, "null argument");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    int n = c->ev_used - 1;
    if (n < 0) n = 0;
    for (int i = 0; i < n && i < capacity; ++i) CU(cudaEventElapsedTime(&ms[i], c->ev[i], c->ev[i + 1]));
    return n;
}

// ---- host-side tail of the reference ---------------------------------------------------------------

int yolo_b200_draw_rectangles(uint16_t *frame, int h, int w, const yolo_b200_det *dets, int count, int normalised)
{
    if (!frame || (!dets && count > 0) || h < 1 || w < 1) return fail(E_ARG, "bad argument");
    for (int i = 0; i < count; ++i) {
        const yolo_b200_det &d = dets[i];
        int x1 = (int)(normalised ? d.x1 * w : d.x1), x2 = (int)(normalised ? d.x2 * w : d.x2);
        int y1 = (int)(normalised ? d.y1 * h : d.y1), y2 = (int)(normalised ? d.y2 * h : d.y2);
        x1 = x1 < 0 ? 0 : (x1 >= w ? w - 1 : x1); x2 = x2 < 0 ? 0 : (x2 >= w ? w - 1 : x2);
        y1 = y1 < 0 ? 0 : (y1 >= h ? h - 1 : y1); y2 = y2 < 0 ? 0 : (y2 >= h ? h - 1 : y2);
        uint16_t px = d.cls == 0 ? 0x000f : 0x00f0;          // red / green, yolo_forward.c:1152-1153,1165-1166
        for (int x = x1; x <= x2; ++x) { frame[(size_t)y1 * w + x] = px; frame[(size_t)y2 * w + x] = px; }
        for (int y = y1; y <= y2; ++y) { frame[(size_t)y * w + x1] = px; frame[(size_t)y * w + x2] = px; }
    }
    return 0;
}

int yolo_b200_set_default_context(yolo_b200_ctx *c)
{
    std::lock_guard<std::mutex> g(g_default_mu);
    g_default_ctx = c;
    return 0;
}

void yolo_forward(const char TRow, const char TCol, const char Tr, const char Tc, const char Tm, const char Tn,
                  short int *camera, int *vga)
{
    (void)Tm; (void)Tn;
    yolo_b200_ctx *c;
    { std::lock_guard<std::mutex> g(g_default_mu); c = g_default_ctx; }
    if (!c) { fail(E_STATE, "yolo_forward: no default context (yolo_b200_set_default_context)"); fprintf(stderr, "%s\n", g_err); return; }
    if (TRow != Tr + 2 || TCol != Tc + 2) { fail(E_ARG, "yolo_forward: TRow/TCol must be Tr+2/Tc+2"); fprintf(stderr, "%s\n", g_err); return; }
    if (!camera || !vga) { fail(E_ARG, "yolo_forward: null frame buffer"); fprintf(stderr, "%s\n", g_err); return; }
    const int W = 320, H = 240;                               // yolo_forward.c:1194-1197
    std::vector<yolo_b200_det> dets(c->prm.max_det);
    int32_t count = 0;
    if (yolo_b200_forward_rgb444(c, (const uint16_t *)camera, 1, H, W, dets.data(), &count)) { fprintf(stderr, "%s\n", g_err); return; }
    if (count > c->prm.max_det) count = c->prm.max_det;
    yolo_b200_draw_rectangles((uint16_t *)camera, H, W, dets.data(), count, c->prm.head_mode == YOLO_B200_HEAD_PYTHON);
    memcpy(vga, camera, (size_t)76800 * 2);                   // yolo_forward.c:1281
}

}  // extern "C"
#pragma GCC visibility pop
