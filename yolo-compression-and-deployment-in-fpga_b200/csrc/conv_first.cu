// conv_first.cu — the network's first layer: 3x3/stride-1/pad-1 convolution of the NHWC4 int8 input (R,G,B,0 per pixel)
// to <= 16 channels, with requantisation, leaky-ReLU and the optional 2x2 max-pool fused.
//
// Replaces first_conv (c_embedding/yolo_forward.c:269-418) and conv1 + tracker + pool (models/slim_yolo_v2.py:220-231).
// K = 27 is far too thin for the tcgen05 path (an M=128 MMA costs >= ~43 cycles whatever N and K are), and the layer is
// bound by instruction issue and shared-memory traffic, not by math.  It runs on warp-level integer MMAs
// (mma.sync.m16n8k32.s8) because their A fragment needs NO im2col staging at all: with K ordered (tap, channel) a thread's
// 32-bit A register is exactly one NHWC4 pixel word of the haloed input tile, i.e. one tap.  K = 36 = 9 taps x 4 bytes is
// covered by one k32 step (taps 0-7) and one k16 step (tap 8 + three zero-weight taps).
//
// Pooled variant: a warp owns 2 pooled rows x 8 pooled columns and runs four M=16 tiles, one per position (dy,dx) of the
// 2x2 window, so the four members of a pooled pixel are the same accumulator slot of the four tiles and the max is taken
// in registers (requantisation is monotone: max-then-requantise == requantise-then-max, slim_yolo_v2.py:229-231).
// Output channels are assigned to the two N=8 tiles so that thread t of a quad ends up with channels 4t..4t+3 of its
// pixel: one 32-bit store per pixel, 16 contiguous bytes per quad, 128 per warp row.
#include "kernels.h"
#include "epilogue.cuh"
#include "ptx.cuh"

namespace yb {

struct FirstParams {
    const int8_t *in;          // [n][H][W][4]  (RGB444 = false)
    const uint16_t *in16;      // [n][H][W] 0x0BGR camera pixels (RGB444 = true): quantised on the fly through the LUT
    const int *lut;            // 4096 packed (R,G,B,0) words = pixel_norm_quantize for every code (yolo_forward.c:57-85)
    const uint8_t *in8;        // [n][H][W][3] BGR bytes (SRC = 2): BaseTransform-without-resize + tracker quantiser through lut8
    const uint8_t *lut8;       // [3][256]: R (from byte 2), G, B
    int n_img, H, W;
    int OH, OW;
    size_t out_img_bytes;      // OH * OW * cs_out
    int cs_out;                // 16; WIDE: any multiple of 16 (the kernel then writes the 16 channels co0 .. co0 + 15 of every pixel)
    int co0;                   // first output channel of this pass
    int xsplit;                // POOL, cs_out == 16: output rows are stored split by x parity, [even pixels][odd pixels] (conv_rp.cu reads them)
    const int8_t *wgt;         // [cout_pad][9][4]
    const int *bias_sh;
    LayerQ q;
    EpiConst k;
    int8_t *out;
    unsigned *ovf;
};

constexpr int F_TW = 32, F_TH = 16;                 // CTA tile, pre-pool pixels
constexpr int F_PITCH = 49;                         // words per halo row (>= F_TW + 2; 49 = 17 mod 32 keeps the tap rows on disjoint banks)
constexpr int F_HROWS = F_TH + 2;
constexpr int F_THREADS = 256;

__device__ __forceinline__ void mma_s8_k32(int (&c)[4], unsigned a0, unsigned a1, unsigned a2, unsigned a3, unsigned b0, unsigned b1)
{
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma_s8_k16(int (&c)[4], unsigned a0, unsigned a1, unsigned b0)
{
    asm volatile("mma.sync.aligned.m16n8k16.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]) : "r"(a0), "r"(a1), "r"(b0));
}

// POOL: tile = 32 x 16 pre-pool pixels -> 16 x 8 pooled; warp w = pooled rows 2*(w>>1), +1 and pooled columns 8*(w&1)..+7.
// !POOL: tile = 32 x 16 pixels; warp w = rows 2w, 2w+1 and four column groups of 8 (four M=16 tiles, rows g / g+8 = the two rows).
// SRC: 0 = int8 NHWC4; 1 = RGB444 camera frames: the RGB444 -> int8 quantiser (camera_to_inpBuf + pixel_norm_quantize,
// yolo_forward.c:57-123) is applied while the halo tile is staged, one lookup in the 4096-entry table per pixel;
// 2 = uint8 BGR image (three 256-entry tables, see quantize.cu).
//
// Persistent and software-pipelined: a CTA loads the table(s), its B fragments and biases once and then walks tiles
// blockIdx.x, +gridDim.x, ...  The halo tile lives in two shared-memory buffers: the global load of tile k+1 is issued
// before the MMAs and the epilogue of tile k (its latency hides behind that work; what stays live is the raw pixels and a
// validity word per thread), is converted through the table into the other buffer afterwards, and ONE barrier per tile
// separates the generations.  The halo is fetched as aligned pixel QUADS (columns x0-4 .. x0+35, 10 quads per row, 180 per
// tile: one per thread), so an RGB444 quad is one 64-bit load (W % 4 == 0 and an aligned frame pointer are required, see
// conv3x3_first_supported / conv3x3_first_src_ok); tile coordinates advance incrementally (no per-tile divisions).
constexpr int F_QUADS_ROW = (F_TW + 8) / 4;                           // 10
constexpr int F_NQUAD = F_HROWS * F_QUADS_ROW;                        // 180 <= F_THREADS
constexpr int F_COL0 = 3;                                             // halo column of x = x0 - 1
static_assert(F_NQUAD <= F_THREADS && 4 * F_QUADS_ROW <= F_PITCH, "one quad per thread");

__device__ __forceinline__ int keep(int v) { asm volatile("" : "+r"(v)); return v; }   // stops the compiler re-deriving v from tid per tile

template <bool POOL, int EPI, bool ACT, int SRC, bool WIDE = false>
__global__ void __launch_bounds__(F_THREADS, 4) conv3x3_first_kernel(const FirstParams p)
{
    // pixel stride of the output map in bytes: 16 for slim_yolo_v2's first layer (compile-time constant); WIDE = a first layer
    // with more than 16 output channels (darknet19: 32), written in passes of 16 channels
    const int PX = WIDE ? p.cs_out : 16;
    pdl_launch_dependents();
    constexpr bool RGB444 = SRC == 1, U8 = SRC == 2;
    constexpr int RAWN = RGB444 ? 2 : U8 ? 3 : 4;                     // 32-bit words per pixel quad
    // fp32 epilogues: the accumulators start at the bit pattern of 1.5 * 2^23, so that read as fp32 they are MAGIC + sum
    // (|sum| <= 27 * 128 * 128 < 2^22) and the epilogue needs no int -> float conversion (requant_f_rne_x2, PRE)
    constexpr bool PRE = EPI == EPI_F_RNE || EPI == EPI_F_RNE_NOHI;
    constexpr int ACC0 = PRE ? YB_MAGIC_BITS : 0;
    __shared__ unsigned s_in[2][F_HROWS * F_PITCH];                   // column c of a row <-> x = x0 - 4 + c
    __shared__ unsigned s_lut[RGB444 ? 4097 : U8 ? 192 : 1];          // RGB444: entry 4096 = 0 = "outside the image"
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;

    if (RGB444) { for (int i = threadIdx.x; i < 4096; i += F_THREADS) s_lut[i] = (unsigned)__ldg(p.lut + i); if (threadIdx.x == 0) s_lut[4096] = 0u; }
    if (U8) for (int i = threadIdx.x; i < 192; i += F_THREADS) s_lut[i] = __ldg(reinterpret_cast<const unsigned *>(p.lut8) + i);
    const unsigned char *s_lut8 = reinterpret_cast<const unsigned char *>(s_lut);

    // B fragments.  N-tile n, column c <-> output channel 4*(c>>1) + 2*n + (c&1), so that the C fragment of thread t
    // (columns 2t, 2t+1 of both tiles) is channels 4t .. 4t+3.
    const unsigned *gw = reinterpret_cast<const unsigned *>(p.wgt) + (WIDE ? p.co0 * 9 : 0);       // word (o*9 + tap) = the 4 channel bytes of one tap
    unsigned b0[2], b1[2], b2[2];
#pragma unroll
    for (int n = 0; n < 2; ++n) {
        const int o = 4 * (g >> 1) + 2 * n + (g & 1);
        b0[n] = __ldg(gw + o * 9 + t);             // k32 step, k = 4t..4t+3    : tap t
        b1[n] = __ldg(gw + o * 9 + 4 + t);         //           k = 16+4t..     : tap 4+t
        b2[n] = t == 0 ? __ldg(gw + o * 9 + 8) : 0u;   // k16 step: tap 8, then three zero taps
    }
    const int4 bias = *reinterpret_cast<const int4 *>(p.bias_sh + (WIDE ? p.co0 : 0) + 4 * t);
    int4 bw = bias;
    if (EPI == EPI_F_RNE || EPI == EPI_F_RNE_NOHI)
        bw = make_int4(__float_as_int((float)bias.x), __float_as_int((float)bias.y), __float_as_int((float)bias.z), __float_as_int((float)bias.w));

    // Word offsets of this thread's A registers inside a halo buffer: tile-invariant origin + tap t, tap 4+t, tap 8
    const int a_org = POOL ? (4 * (warp >> 1)) * F_PITCH + 2 * (8 * (warp & 1) + g) + F_COL0
                           : (2 * warp) * F_PITCH + g + F_COL0;
    const int o_a = keep(a_org + (t / 3) * F_PITCH + (t % 3));
    const int o_b = keep(a_org + ((4 + t) / 3) * F_PITCH + ((4 + t) % 3));
    const int o_c = keep(a_org + 2 * F_PITCH + 2);
    // this thread's output pixel inside a tile (rows oy_t, oy_t + 1; column ox_t [+ 8 cg]) and its byte offset
    const int oy_t = keep(POOL ? 2 * (warp >> 1) : 2 * warp), ox_t = keep(POOL ? 8 * (warp & 1) + g : g);
    // x-split rows (POOL only): pooled pixel x lives at (x & 1) * OW/2 + (x >> 1) of its row; a tile's 16 pooled columns start at an
    // even x, so the split is a per-thread constant
    const int ox_s = (POOL && p.xsplit) ? (ox_t & 1) * (p.OW >> 1) + (ox_t >> 1) : ox_t;
    const int o_thr = keep((oy_t * (POOL ? p.OW : p.W) + ox_s) * PX + 4 * t + (WIDE ? p.co0 : 0));
    unsigned ovf = 0;

    const int tiles_x = (p.W + F_TW - 1) / F_TW, tiles_y = (p.H + F_TH - 1) / F_TH;
    const int tiles_img = tiles_x * tiles_y;
    // one grid stride, decomposed into (images, tile rows, tile columns)
    const int s_img = (int)gridDim.x / tiles_img;
    const int s_y = ((int)gridDim.x - s_img * tiles_img) / tiles_x, s_x = (int)gridDim.x - s_img * tiles_img - s_y * tiles_x;
    int img = (int)blockIdx.x / tiles_img;
    int ty = ((int)blockIdx.x - img * tiles_img) / tiles_x, tx = (int)blockIdx.x - img * tiles_img - ty * tiles_x;

    // this thread's halo quad: halo row tid / 10, columns 4 (tid % 10) .. +3
    const bool has_quad = threadIdx.x < F_NQUAD;
    const int q_hy = has_quad ? (int)threadIdx.x / F_QUADS_ROW : -0x1000000;  // no quad: fails the row test
    const int q_hx = 4 * ((int)threadIdx.x % F_QUADS_ROW);
    const int q_goff = keep(has_quad ? q_hy * p.W + q_hx : 0);               // pixel offset from the halo's top-left corner
    const int q_soff = keep(has_quad ? q_hy * F_PITCH + q_hx : 0);
    unsigned raw[RAWN];
    unsigned oob = 0;              // RGB444: 0x1000 in both half-words when the quad lies outside the image (table entry 4096 = 0)
    auto fetch = [&](int im, int y0, int x0) {
        const int y = y0 - 1 + q_hy, x = x0 - 4 + q_hx;
        const bool ok = (unsigned)y < (unsigned)p.H && (unsigned)x < (unsigned)p.W;   // W % 4 == 0: a quad is all in or all out
        const int e = (im * p.H + (y0 - 1)) * p.W + (x0 - 4) + q_goff;  // pixel index (host: n*H*W < 2^31)
#pragma unroll
        for (int i = 0; i < RAWN; ++i) raw[i] = 0u;
        if (RGB444) {
            if (ok) { const uint2 v = __ldg(reinterpret_cast<const uint2 *>(p.in16 + e)); raw[0] = v.x; raw[1] = v.y; }
            oob = ok ? 0u : 0x10001000u;
        } else if (U8) {
            if (ok) { const unsigned *px = reinterpret_cast<const unsigned *>(p.in8 + 3 * (size_t)e); raw[0] = __ldg(px); raw[1] = __ldg(px + 1); raw[2] = __ldg(px + 2); }
            oob = ok ? 0u : 1u;
        } else {
            if (ok) { const uint4 v = __ldg(reinterpret_cast<const uint4 *>(reinterpret_cast<const unsigned *>(p.in) + e)); raw[0] = v.x; raw[1] = v.y; raw[2] = v.z; raw[3] = v.w; }
        }
    };
    // table lookups + stores of the fetched quad; zero outside the image (= the convolution's zero padding)
    auto u8px = [&](unsigned c) {                                      // c = B | G << 8 | R << 16
        return (unsigned)s_lut8[(c >> 16) & 255u] | ((unsigned)s_lut8[256 + ((c >> 8) & 255u)] << 8) | ((unsigned)s_lut8[512 + (c & 255u)] << 16);
    };
    auto stage = [&](unsigned *dst) {
        if (has_quad) {
            unsigned v[4];
            if (RGB444) {
                const unsigned r0 = (raw[0] & 0x0fff0fffu) | oob, r1 = (raw[1] & 0x0fff0fffu) | oob;
                v[0] = s_lut[r0 & 0xffffu]; v[1] = s_lut[r0 >> 16]; v[2] = s_lut[r1 & 0xffffu]; v[3] = s_lut[r1 >> 16];
            } else if (U8) {
                // bytes: B0 G0 R0 B1 | G1 R1 B2 G2 | R2 B3 G3 R3
                v[0] = u8px(raw[0]);
                v[1] = u8px((raw[0] >> 24) | (raw[1] << 8));
                v[2] = u8px((raw[1] >> 16) | (raw[2] << 16));
                v[3] = u8px(raw[2] >> 8);
                if (oob) { v[0] = 0u; v[1] = 0u; v[2] = 0u; v[3] = 0u; }
            } else { v[0] = raw[0]; v[1] = raw[1]; v[2] = raw[2]; v[3] = raw[3]; }
            unsigned *d = dst + q_soff;
            d[0] = v[0]; d[1] = v[1]; d[2] = v[2]; d[3] = v[3];
        }
    };
    auto advance = [&](int &im, int &y, int &x) {
        x += s_x; if (x >= tiles_x) { x -= tiles_x; ++y; }
        y += s_y; if (y >= tiles_y) { y -= tiles_y; ++im; }
        im += s_img;
    };

    __syncthreads();                                                   // tables loaded
    pdl_wait();                                                        // the previous kernel is done: the input may be read, the output map written
    fetch(img, ty * F_TH, tx * F_TW);
    stage(s_in[0]);
    __syncthreads();
    int buf = 0;
    while (img < p.n_img) {
        int nimg = img, nty = ty, ntx = tx;
        advance(nimg, nty, ntx);
        const bool has_next = nimg < p.n_img;
        if (has_next) fetch(nimg, nty * F_TH, ntx * F_TW);             // in flight during this tile's MMAs and epilogue
        const unsigned *tile_in = s_in[buf];
        const int x0 = tx * F_TW, y0 = ty * F_TH;

        if (POOL) {
            int acc[4][2][4];
#pragma unroll
            for (int ph = 0; ph < 4; ++ph)
#pragma unroll
                for (int n = 0; n < 2; ++n)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[ph][n][j] = ACC0;
#pragma unroll
            for (int ph = 0; ph < 4; ++ph) {
                const int dy = ph >> 1, dx = ph & 1;
                // rows g / g+8 of the M=16 tile: pooled pixel (pr0, pc0+g) / (pr0+1, pc0+g), member (dy,dx)
                const unsigned *r0 = tile_in + dy * F_PITCH + dx;
                const unsigned *r1 = r0 + 2 * F_PITCH;
                const unsigned a0 = r0[o_a], a1 = r1[o_a], a2 = r0[o_b], a3 = r1[o_b], a4 = r0[o_c], a5 = r1[o_c];
#pragma unroll
                for (int n = 0; n < 2; ++n) {
                    mma_s8_k32(acc[ph][n], a0, a1, a2, a3, b0[n], b1[n]);
                    mma_s8_k16(acc[ph][n], a4, a5, b2[n]);
                }
            }
            // this thread's 4 channels of pooled pixel (oy, ox)
            int8_t *out_px = p.out + (size_t)img * p.out_img_bytes + ((((y0 >> 1) * p.OW + (p.xsplit ? x0 >> 2 : x0 >> 1)) * PX) + o_thr);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                int m[4];
#pragma unroll
                for (int n = 0; n < 2; ++n)
#pragma unroll
                    for (int c = 0; c < 2; ++c)
                        m[2 * n + c] = max(max(acc[0][n][2 * h + c], acc[1][n][2 * h + c]), max(acc[2][n][2 * h + c], acc[3][n][2 * h + c]));
                const int oy = (y0 >> 1) + oy_t + h, ox = (x0 >> 1) + ox_t;
                const bool valid = oy < p.OH && ox < p.OW;
                const unsigned w = requant4v<EPI, ACT, FirstParams, PRE>(m, bw, p, ovf, valid);
                if (valid) *reinterpret_cast<unsigned *>(out_px + h * p.OW * PX) = w;
            }
        } else {
            int8_t *out_px = p.out + (size_t)img * p.out_img_bytes + (((y0 * p.W + x0) * PX) + o_thr);
#pragma unroll
            for (int cg = 0; cg < 4; ++cg) {
                int acc[2][4];
#pragma unroll
                for (int n = 0; n < 2; ++n)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[n][j] = ACC0;
                const unsigned *r0 = tile_in + 8 * cg;                     // rows 2 warp, 2 warp + 1 of the tile
                const unsigned *r1 = r0 + F_PITCH;
                const unsigned a0 = r0[o_a], a1 = r1[o_a], a2 = r0[o_b], a3 = r1[o_b], a4 = r0[o_c], a5 = r1[o_c];
#pragma unroll
                for (int n = 0; n < 2; ++n) {
                    mma_s8_k32(acc[n], a0, a1, a2, a3, b0[n], b1[n]);
                    mma_s8_k16(acc[n], a4, a5, b2[n]);
                }
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int m[4] = { acc[0][2 * h], acc[0][2 * h + 1], acc[1][2 * h], acc[1][2 * h + 1] };
                    const int y = y0 + oy_t + h, x = x0 + 8 * cg + ox_t;
                    const bool valid = y < p.H && x < p.W;
                    const unsigned w = requant4v<EPI, ACT, FirstParams, PRE>(m, bw, p, ovf, valid);
                    if (valid) *reinterpret_cast<unsigned *>(out_px + (h * p.W + 8 * cg) * PX) = w;
                }
            }
        }

        if (has_next) stage(s_in[buf ^ 1]);
        __syncthreads();                                               // tile k+1 staged; tile k's buffer free for tile k+2
        buf ^= 1; img = nimg; ty = nty; tx = ntx;
    }
    if (p.q.contract == CONTRACT_P) {
        ovf = __reduce_add_sync(0xffffffffu, ovf);
        if (lane == 0 && ovf) atomicAdd(p.ovf, ovf);
    }
}

bool conv3x3_first_supported(const ConvArgs &a)
{
    if (a.cs_in != 4 || a.cs_out % 16 || a.cs_out > 64 || a.w_rows < a.cs_out) return false;   // 16 channels per pass
    if (a.q.pool && (a.H < 2 || a.W < 2)) return false;
    if (a.W % 4) return false;                                                     // the halo is fetched as aligned pixel quads
    if ((long long)a.n * a.H * a.W >= (1ll << 31) - (1ll << 20)) return false;     // 32-bit pixel offsets in the halo fetch
    return true;
}

// alignment the quad loads need from the source pointer (frames are W*H pixels with W % 4 == 0, so every quad inherits it)
bool conv3x3_first_src_ok(InKind src_kind, const void *src)
{
    return ((uintptr_t)src % (src_kind == IN_RGB444 ? 8 : src_kind == IN_BGR ? 4 : 16)) == 0;
}

template <bool POOL, int EPI, int SRC, bool WIDE = false>
static cudaError_t launch_first3(const FirstParams &p, cudaStream_t st)
{
    const long long total = (long long)((p.W + F_TW - 1) / F_TW) * ((p.H + F_TH - 1) / F_TH) * p.n_img;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // persistent grid = exactly the CTAs that are resident at once
    int per_sm = 0;
    cudaError_t e = p.q.activ ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, conv3x3_first_kernel<POOL, EPI, true, SRC, WIDE>, F_THREADS, 0)
                              : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, conv3x3_first_kernel<POOL, EPI, false, SRC, WIDE>, F_THREADS, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    const long long cap = (long long)sms * per_sm;
    const int grid = (int)(total < cap ? total : cap);
    if (p.q.activ) return launch_pdl(conv3x3_first_kernel<POOL, EPI, true, SRC, WIDE>, dim3(grid), dim3(F_THREADS), 0, st, p);
    return launch_pdl(conv3x3_first_kernel<POOL, EPI, false, SRC, WIDE>, dim3(grid), dim3(F_THREADS), 0, st, p);
}

template <bool POOL, int EPI>
static cudaError_t launch_first2(const FirstParams &p, cudaStream_t st)
{
    if (p.cs_out != 16) {
        // wider first layers (darknet19's 3 -> 32): one pass per 16 output channels over the same input
        FirstParams q = p;
        for (q.co0 = 0; q.co0 < p.cs_out; q.co0 += 16) {
            cudaError_t e = p.in16 ? launch_first3<POOL, EPI, IN_RGB444, true>(q, st) : p.in8 ? launch_first3<POOL, EPI, IN_BGR, true>(q, st) : launch_first3<POOL, EPI, IN_INT8, true>(q, st);
            if (e != cudaSuccess) return e;
        }
        return cudaSuccess;
    }
    if (p.in16) return launch_first3<POOL, EPI, IN_RGB444>(p, st);
    if (p.in8) return launch_first3<POOL, EPI, IN_BGR>(p, st);
    return launch_first3<POOL, EPI, IN_INT8>(p, st);
}

template <bool POOL>
static cudaError_t launch_first(const ConvArgs &a, FirstParams &p, cudaStream_t st)
{
    switch (epi_mode_for(a, &p.k)) {
    case EPI_F_RNE:      return launch_first2<POOL, EPI_F_RNE>(p, st);
    case EPI_F_RNE_NOHI: return launch_first2<POOL, EPI_F_RNE_NOHI>(p, st);
    case EPI_P:          return launch_first2<POOL, EPI_P>(p, st);
    default:             return launch_first2<POOL, EPI_GENERIC>(p, st);
    }
}

// src_kind IN_RGB444 / IN_BGR: fused RGB444 / uint8-BGR front end (a.in is ignored); lut = the context's table for that source
cudaError_t conv3x3_first(const ConvArgs &a, cudaStream_t st, InKind src_kind, const void *src, const void *lut)
{
    if (a.n == 0) return cudaSuccess;
    if (!conv3x3_first_supported(a)) return cudaErrorInvalidValue;
    // the benchmark geometries (pooled, 16 channels, pooled width >= 128) run on the tcgen05 kernel of conv_fs.cu
    if (conv3x3_fs_supported(a, src_kind, src_kind != IN_INT8 ? src : (const void *)a.in))
        return conv3x3_fs(a, st, src_kind, src_kind != IN_INT8 ? src : (const void *)a.in, lut);
    FirstParams p;
    memset(&p, 0, sizeof p);
    p.in = a.in; p.n_img = a.n; p.H = a.H; p.W = a.W;
    if (src_kind == IN_RGB444) { p.in16 = (const uint16_t *)src; p.lut = (const int *)lut; }
    else if (src_kind == IN_BGR) { p.in8 = (const uint8_t *)src; p.lut8 = (const uint8_t *)lut; }
    // a pixel quad = 8 bytes of RGB444, 12 of BGR bytes (three word loads), 16 of NHWC4
    if (!conv3x3_first_src_ok(src_kind, src_kind != IN_INT8 ? src : (const void *)a.in)) return cudaErrorInvalidValue;
    p.OH = a.q.pool ? a.H / 2 : a.H; p.OW = a.q.pool ? a.W / 2 : a.W;
    p.out_img_bytes = (size_t)p.OH * p.OW * a.cs_out;
    p.cs_out = a.cs_out; p.wgt = a.wgt; p.bias_sh = a.bias_sh; p.q = a.q; p.out = a.out; p.ovf = a.ovf;
    if (a.out_xsplit) {
        if (!a.q.pool || a.cs_out != 16 || (p.OW & 1)) return cudaErrorInvalidValue;
        p.xsplit = 1;
    }
    return a.q.pool ? launch_first<true>(a, p, st) : launch_first<false>(a, p, st);
}

}  // namespace yb
