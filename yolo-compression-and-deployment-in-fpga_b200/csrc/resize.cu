// Bilinear resize of uint8 HxWx3 images in front of the first layer: the GPU replacement of
// `cv2.resize(image, (size[1], size[0]))` in base_transform (reference data/__init__.py:36), bit-exact with OpenCV's 8-bit
// INTER_LINEAR (11-bit fixed-point taps, horizontal pass at scale 2^11, vertical pass `((b*(H>>4))>>16)`, `(+2)>>2`).
// The per-column / per-row taps and weights are computed once on the host in the float/double arithmetic OpenCV uses
// (resize_axis_table) and kept in two small device tables; exact 2x decimation, where OpenCV switches to the 2x2 area
// mean, falls out of the same formula (both weights are 1024 and the shifts are exact), so there is one kernel.
//
// HBM-bound byte work: per output pixel 12 source bytes (mostly L1/L2 hits: neighbouring outputs share taps) and 3 output
// bytes.  What limits such a kernel is the number of 128-byte lines each load instruction touches, so the source is read
// through aligned 32-bit words (see resize_row_taps) and a warp's 96 output bytes leave as 24 word stores.
// History (256 frames 480x640 -> 416x416): four pixels per thread with byte loads 0.344 ms (every byte load touched 5-6
// lines); one pixel per thread numbered flat over the batch with word loads 0.40 ms -- ncu: 226 instructions per pixel,
// issue-bound on the 64-bit index divisions; one row per CTA iteration (grid-stride) with DP2A / high-multiply
// arithmetic 0.376 ms -- still 200 instructions per 32-pixel chunk, 72 of them row bookkeeping repeated by every warp and
// 24 of them 64-bit addresses of the clamped word loads; this version (one warp per run of contiguous rows, clamping only
// in the rows that can reach the end of the buffer) 0.207 ms at 47 registers / 40 resident warps per SM (98 instructions per
// chunk, 57 % issue utilisation, long-scoreboard stalls: latency-bound), 0.193 ms (ncu: profiles/resize_r1_ncu.txt) =
// 1.91 TB/s of algorithmic bytes capped at 40 registers / 48 warps (what ships).  Measured slower: the chunk loop unrolled
// by two (54 registers, 32 warps: 0.233 ms), a 32-register cap (64 warps, spills: 0.226 ms).
#include "kernels.h"

#include <cmath>
#include <vector>

namespace yb {

void resize_axis_table(int src, int dst, bool clamp_weights, int index_scale, int4 *out)
{
    // cv::resize: inv_scale = (double)dst/src; cv::hal::resize: scale = 1./inv_scale
    volatile double inv_scale = (double)dst / (double)src;
    volatile double scale = 1.0 / inv_scale;
    for (int d = 0; d < dst; ++d) {
        volatile double t = (d + 0.5) * scale;                // volatile: no fused multiply-add on the host
        float f = (float)(t - 0.5);
        int s = (int)floorf(f);
        f -= (float)s;
        if (clamp_weights) {                                   // horizontal pass: the tap is re-anchored at the border
            if (s < 0) { s = 0; f = 0.f; }
            if (s >= src - 1) { s = src - 1; f = 0.f; }
        }
        const int c0 = (int)lrintf((1.f - f) * 2048.f), c1 = (int)lrintf(f * 2048.f);    // saturate_cast<short>: RNE
        int i0 = s < 0 ? 0 : (s > src - 1 ? src - 1 : s);
        int i1 = s + 1 < 0 ? 0 : (s + 1 > src - 1 ? src - 1 : s + 1);
        out[d] = make_int4(i0 * index_scale, i1 * index_scale, c0, c1);
    }
}

// One source row's contribution: the six bytes (tap 0 = bytes 0..2, tap 1 = bytes 3..5) that start `off` bytes into a
// word-aligned view of the row, fetched as three aligned 32-bit words and realigned with funnel shifts (a warp's lanes
// are ~4.6 bytes apart for 640 -> 416, so a word load touches two 128-byte lines).  CLAMP (only the rows whose windows
// could reach past the end of the buffer, i.e. the last source rows of the last image): byte loads with indices clamped
// to `lim`, the last byte of the buffer relative to this row; a clamped byte only ever supplies a zero-weight value
// (tap 1 of a right-border pixel).  compute-sanitizer memcheck runs clean on the GPU tests with exact-size allocations.
template <bool CLAMP>
__device__ __forceinline__ void resize_row_taps(const unsigned char *__restrict__ rowb, unsigned off, unsigned lim, unsigned &lo, unsigned &hi)
{
    if (CLAMP) {
        // byte loads, indices clamped to the last byte of the buffer (`lim`, relative to rowb)
        lo = 0; hi = 0;
#pragma unroll
        for (unsigned k = 0; k < 4; ++k) lo |= (unsigned)__ldg(rowb + min(off + k, lim)) << (8 * k);
#pragma unroll
        for (unsigned k = 0; k < 2; ++k) hi |= (unsigned)__ldg(rowb + min(off + 4 + k, lim)) << (8 * k);
    } else {
        const unsigned sh = (off & 3u) * 8u;
        const unsigned *a = reinterpret_cast<const unsigned *>(rowb + (off & ~3u));     // one address, three immediates
        const unsigned w0 = __ldg(a), w1 = __ldg(a + 1), w2 = __ldg(a + 2);
        lo = __funnelshift_r(w0, w1, sh);          // bytes off .. off+3
        hi = __funnelshift_r(w1, w2, sh);          // bytes off+4 .. off+7
    }
}

// a01 = weight0 | weight1 << 16 (units of 1/2048), B0/B1 = row weights << 16.  Per channel: the horizontal pass of one
// row is one PRMT (tap 0 and tap 1 bytes side by side) + one unsigned DP2A; `(b * (h >> 4)) >> 16` is a high multiply.
// The window of a row is lo | hi << 32: tap 0 from byte 0, tap 1 from byte TAP1 (3 for packed 3-byte pixels, 4 for one
// 32-bit word per pixel).  RGB: the pixels are R, G, B, so output channel ch (B, G, R) comes from byte 2 - ch of a tap.
template <bool RGB = false, unsigned TAP1 = 3>
__device__ __forceinline__ unsigned resize_combine(unsigned lo0, unsigned hi0, unsigned lo1, unsigned hi1, unsigned a01, unsigned B0, unsigned B1)
{
    unsigned o[3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        const unsigned c = RGB ? 2u - (unsigned)ch : (unsigned)ch;
        const unsigned sel = c | ((TAP1 + c) << 4);                              // bytes c and TAP1 + c of the 8-byte window
        const unsigned h0 = __dp2a_lo(a01, __byte_perm(lo0, hi0, sel), 0u);    // horizontal pass, scale 2^11
        const unsigned h1 = __dp2a_lo(a01, __byte_perm(lo1, hi1, sel), 0u);
        o[ch] = (__umulhi(B0, h0 >> 4) + __umulhi(B1, h1 >> 4) + 2u) >> 2;      // <= 255 by construction
    }
    return o[0] | (o[1] << 8) | (o[2] << 16);
}

// The store of one 32-pixel chunk (v = B | G << 8 | R << 16 of this lane's pixel).  WORD_STORE: the 32 three-byte pixels
// of a full warp are regrouped by two shuffles into 24 aligned 32-bit stores (output word j = bytes 4j .. 4j+3 of the
// chunk = pixels p = 4j/3 and p + 1 from byte rsh/8 of p); partial chunks and other geometries store bytes.
template <bool WORD_STORE>
__device__ __forceinline__ void resize_store(unsigned v, bool live, int dx0, int dx, int dw, uint8_t *__restrict__ drow, int lane, int p, unsigned rsh)
{
    if (WORD_STORE && dx0 + 32 <= dw) {
        const unsigned va = __shfl_sync(0xffffffffu, v, p & 31), vb = __shfl_sync(0xffffffffu, v, (p + 1) & 31);
        const unsigned word = __funnelshift_r(va | (vb << 24), vb >> 8, rsh);
        if (lane < 24) reinterpret_cast<unsigned *>(drow)[(dx0 >> 5) * 24 + lane] = word;
    } else if (live) {
        uint8_t *o = drow + (size_t)dx * 3;
        o[0] = (uint8_t)v; o[1] = (uint8_t)(v >> 8); o[2] = (uint8_t)(v >> 16);
    }
}

// One output row of the batch: one thread = one output pixel, a warp = 32 consecutive pixels = 96 contiguous output bytes.
// RGB: the source pixels are R, G, B (resize_combine).
// GROUP_LOADS (the pitched instantiations' unclamped rows): the six words of both source rows are loaded in one asm
// statement before any is used.  Left to itself, ptxas schedules the pitched loop at its 48-register budget with the second
// row's loads after the first row's funnel shifts, so every chunk waits for two load latencies in turn (0.234 against
// 0.205 ms for the same loop in the ragged instantiation).
template <bool WORD_STORE, bool CLAMP, bool RGB, bool GROUP_LOADS = false>
__device__ __forceinline__ void resize_one_row(const unsigned char *__restrict__ r0, const unsigned char *__restrict__ r1,
                                               unsigned d0, unsigned d1, unsigned lim0, unsigned lim1, unsigned B0, unsigned B1,
                                               const int2 *__restrict__ xtab, uint8_t *__restrict__ drow, int dw,
                                               int lane, int warp, int nwarps, int p, unsigned rsh)
{
    for (int dx0 = warp * 32; dx0 < dw; dx0 += nwarps * 32) {
        const int dx = dx0 + lane;
        const bool live = dx < dw;
        unsigned v = 0;
        if (live) {
            const int2 xt = __ldg(xtab + dx);
            unsigned lo0, hi0, lo1, hi1;
            if constexpr (GROUP_LOADS && !CLAMP) {
                const unsigned off0 = (unsigned)xt.x + d0, off1 = (unsigned)xt.x + d1;
                const unsigned char *a0 = r0 + (off0 & ~3u), *a1 = r1 + (off1 & ~3u);
                unsigned w0, w1, w2, w3, w4, w5;
                asm volatile("ld.global.nc.u32 %0, [%6];\n\tld.global.nc.u32 %1, [%6+4];\n\tld.global.nc.u32 %2, [%6+8];\n\t"
                             "ld.global.nc.u32 %3, [%7];\n\tld.global.nc.u32 %4, [%7+4];\n\tld.global.nc.u32 %5, [%7+8];"
                             : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3), "=r"(w4), "=r"(w5) : "l"(a0), "l"(a1));
                lo0 = __funnelshift_r(w0, w1, (off0 & 3u) * 8u); hi0 = __funnelshift_r(w1, w2, (off0 & 3u) * 8u);
                lo1 = __funnelshift_r(w3, w4, (off1 & 3u) * 8u); hi1 = __funnelshift_r(w4, w5, (off1 & 3u) * 8u);
            } else {
                resize_row_taps<CLAMP>(r0, (unsigned)xt.x + d0, lim0, lo0, hi0);
                resize_row_taps<CLAMP>(r1, (unsigned)xt.x + d1, lim1, lo1, hi1);
            }
            v = resize_combine<RGB>(lo0, hi0, lo1, hi1, (unsigned)xt.y, B0, B1);
        }
        resize_store<WORD_STORE>(v, live, dx0, dx, dw, drow, lane, p, rsh);
    }
}

// ---- YUV sources: cv2.cvtColor(COLOR_YUV2BGR_NV12 / _I420 / _YUYV) fused in front of the resize -------------------------
// OpenCV's 8-bit YUV -> RGB (BT.601 limited range, 20-bit fixed point, modules/imgproc/src/color_yuv.simd.hpp):
//   y = max(Y - 16, 0) * 1220542;  u = U - 128;  v = V - 128
//   R = sat8((y + 2^19 + 1673527 v) >> 20);  G = sat8((y + 2^19 - 852492 v - 409993 u) >> 20);  B = sat8((y + 2^19 + 2116026 u) >> 20)
// with an arithmetic (floor) shift; every sum stays below 6e8 in magnitude, so int32 is exact.  Chroma is nearest:
// one U,V pair per 2x2 block (4:2:0) or per horizontal pixel pair (4:2:2).  Returns B | G << 8 | R << 16.
__device__ __forceinline__ unsigned yuv_to_bgr(unsigned Y, unsigned U, unsigned V)
{
    const int y = max((int)Y - 16, 0) * 1220542 + (1 << 19);
    const int u = (int)U - 128, v = (int)V - 128;
    const int r = (y + 1673527 * v) >> 20, g = (y - 852492 * v - 409993 * u) >> 20, b = (y + 2116026 * u) >> 20;
    return (unsigned)min(max(b, 0), 255) | ((unsigned)min(max(g, 0), 255) << 8) | ((unsigned)min(max(r, 0), 255) << 16);
}

// One source row r of a YUV frame: where its luma and the chroma it uses start (cv2 Mat layouts, no padding).
//   NV12: Y plane sh x sw, then sh/2 rows of sw bytes U,V,U,V...  -> y = row r, u = interleaved chroma row r/2 (v unused)
//   I420: Y plane, U plane (sh/2) x (sw/2), V plane              -> y, u, v = row r, r/2, r/2 of their planes
//   YUYV: sh rows of 2*sw bytes, macropixel Y0 U Y1 V             -> y = row r (u, v unused)
struct YuvRow { const uint8_t *y, *u, *v; };

template <int FMT>
__device__ __forceinline__ YuvRow yuv_row(const uint8_t *frame, unsigned r, int sh, int sw)
{
    const size_t plane = (size_t)sh * sw, c = r >> 1;         // the chroma row is warp-uniform: r is the row's tap
    if (FMT == RS_YUV_NV12) return { frame + (size_t)r * sw, frame + plane + c * sw, nullptr };
    if (FMT == RS_YUV_I420) return { frame + (size_t)r * sw, frame + plane + c * (sw >> 1), frame + plane + plane / 4 + c * (sw >> 1) };
    return { frame + (size_t)r * 2 * sw, nullptr, nullptr };
}

// The same rows of a pitched frame (ResizeLayout): row r of plane p at frame + off[p] + r * pitch[p]; NV12's plane 1 and
// I420's planes 1 and 2 are the chroma rows r/2
template <int FMT>
__device__ __forceinline__ YuvRow yuv_row_pitched(const uint8_t *frame, unsigned r, const ResizeLayout &L)
{
    const unsigned c = r >> 1;
    const uint8_t *y = frame + (L.off[0] + r * L.pitch[0]);
    if (FMT == RS_YUV_NV12) return { y, frame + (L.off[1] + c * L.pitch[1]), nullptr };
    if (FMT == RS_YUV_I420) return { y, frame + (L.off[1] + c * L.pitch[1]), frame + (L.off[2] + c * L.pitch[2]) };
    return { y, nullptr, nullptr };
}

// B | G << 8 | R << 16 of source pixel x of the row
template <int FMT>
__device__ __forceinline__ unsigned yuv_pixel(const YuvRow &row, unsigned x)
{
    if (FMT == RS_YUV_NV12) return yuv_to_bgr(__ldg(row.y + x), __ldg(row.u + (x & ~1u)), __ldg(row.u + (x | 1u)));
    if (FMT == RS_YUV_I420) return yuv_to_bgr(__ldg(row.y + x), __ldg(row.u + (x >> 1)), __ldg(row.v + (x >> 1)));
    const uint8_t *m = row.y + 2 * (x & ~1u);                 // the macropixel of x
    return yuv_to_bgr(__ldg(row.y + 2 * x), __ldg(m + 1), __ldg(m + 3));
}

// A row's 6-byte window in the BGR kernel's form (tap 0 = bytes 0..2, tap 1 = bytes 3..5), converted from YUV.  Tap 1 is
// pixel x0 + 1 except at the right border, where the horizontal table gives tap 1 weight 0 (resize_axis_table re-anchors
// it); there the window takes pixel sw - 1 instead, so no byte left of column 0 or right of column sw - 1 is ever read.
template <int FMT>
__device__ __forceinline__ void yuv_row_taps(const YuvRow &row, unsigned x0, unsigned x1, unsigned &lo, unsigned &hi)
{
    const unsigned p0 = yuv_pixel<FMT>(row, x0), p1 = yuv_pixel<FMT>(row, x1);
    lo = p0 | (p1 << 24);
    hi = p1 >> 8;
}

// The YUV form of resize_u8c3_kernel's row loop: frames of frame_bytes bytes at a uniform stride, the uniform row / column
// tables (xtab's byte offsets are 3 * source column), resize_combine and the same stores.
// Bounds: a source row index comes from ytab (clamped to [0, sh - 1]), a column from xtab (in [0, sw - 1]) or its clamped
// successor, so with sh, sw even where the format subsamples every byte read (luma, chroma row r/2 <= sh/2 - 1, chroma
// column x/2 <= sw/2 - 1) lies inside its own frame, and frames are those of this launch: nothing is read past
// src + n * frame_bytes.  In the chunked host path that is the end of the chunk's landed bytes.  Loads are bytes (a warp's
// lanes are ~1.5 luma bytes apart for 640 -> 416, so each byte load touches one or two 128-byte lines), so there is no
// aligned word that could straddle the end and no clamped-row variant.
// LAYOUT: the frames are pitched as *lay says (rows of the same bytes, at other addresses; the bounds argument holds row by
// row, and nothing is read outside the rows of this launch's frames).
template <bool WORD_STORE, int FMT, bool LAYOUT>
__device__ __forceinline__ void resize_yuv_rows(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, const int2 *__restrict__ xtab,
                                                const int4 *__restrict__ ytab, unsigned row, unsigned row_end, int sh, int sw, int dh, int dw, int lane,
                                                const ResizeLayout *__restrict__ lay)
{
    const int p = (4 * lane) / 3;
    const unsigned rsh = 8u * (unsigned)(4 * lane - 3 * p);
    const size_t plane = (size_t)sh * sw;
    ResizeLayout L{};
    if constexpr (LAYOUT) L = *lay;
    const size_t frame_bytes = LAYOUT ? (size_t)L.stride : FMT == RS_YUV_YUYV ? 2 * plane : plane + plane / 2;
    unsigned dy = row % (unsigned)dh;
    const uint8_t *frame = src + (size_t)(row / (unsigned)dh) * frame_bytes;
    uint8_t *drow = dst + (size_t)row * dw * 3;
    for (; row < row_end; ++row) {
        const int4 yt = __ldg(ytab + dy);
        const YuvRow r0 = LAYOUT ? yuv_row_pitched<FMT>(frame, (unsigned)yt.x, L) : yuv_row<FMT>(frame, (unsigned)yt.x, sh, sw);
        const YuvRow r1 = LAYOUT ? yuv_row_pitched<FMT>(frame, (unsigned)yt.y, L) : yuv_row<FMT>(frame, (unsigned)yt.y, sh, sw);
        for (int dx0 = 0; dx0 < dw; dx0 += 32) {
            const int dx = dx0 + lane;
            const bool live = dx < dw;
            unsigned v = 0;
            if (live) {
                const int2 xt = __ldg(xtab + dx);
                const unsigned x0 = (unsigned)xt.x / 3u, x1 = min(x0 + 1u, (unsigned)sw - 1u);
                unsigned lo0, hi0, lo1, hi1;
                yuv_row_taps<FMT>(r0, x0, x1, lo0, hi0);
                yuv_row_taps<FMT>(r1, x0, x1, lo1, hi1);
                v = resize_combine(lo0, hi0, lo1, hi1, (unsigned)xt.y, (unsigned)yt.z, (unsigned)yt.w);
            }
            resize_store<WORD_STORE>(v, live, dx0, dx, dw, drow, lane, p, rsh);
        }
        drow += (size_t)dw * 3;
        if (++dy == (unsigned)dh) { dy = 0; frame += frame_bytes; }
    }
}

// ---- Bayer sources: cv2.cvtColor(COLOR_Bayer**2BGR) fused in front of the resize ---------------------------------------
// OpenCV's default bilinear demosaic.  A pattern is named by the sensor's top-left 2x2 (RGGB: row 0 = R G R G .., row 1 =
// G B G B ..); GRBG flips RGGB's column parity, GBRG its row parity and BGGR both.  At an interior site (1 <= y <= sh - 2,
// 1 <= x <= sw - 2) with N, S, W, E its 4-neighbours and NW, NE, SW, SE its diagonals, the site's own colour is its byte;
// at an R or B site G = (N + S + W + E + 2) >> 2 and the opposite colour is (NW + NE + SW + SE + 2) >> 2; at a G site the
// colour of its horizontal neighbours is (W + E + 1) >> 1 and that of its vertical neighbours (N + S + 1) >> 1.  cv2
// copies column 1 into column 0 and column sw - 2 into sw - 1, then row 1 into row 0 and row sh - 2 into row sh - 1, so
// BGR(y, x) = interior(clamp(y, 1, sh - 2), clamp(x, 1, sw - 2)).

// B | G << 8 | R << 16 of the interior site v[1][1] of a 3x3 window (rows i, columns j of a 4x4 grid from (i0, j0));
// xo, yo: the site's column and row parity counted from an R site
__device__ __forceinline__ unsigned bayer_site(const unsigned (&v)[4][4], int i0, int j0, unsigned xo, unsigned yo)
{
    const int i = i0 + 1, j = j0 + 1;
    const unsigned hs = v[i][j - 1] + v[i][j + 1], vs = v[i - 1][j] + v[i + 1][j];
    const unsigned diag = (v[i - 1][j - 1] + v[i - 1][j + 1] + v[i + 1][j - 1] + v[i + 1][j + 1] + 2u) >> 2;
    const unsigned cross = (hs + vs + 2u) >> 2, hh = (hs + 1u) >> 1, vv = (vs + 1u) >> 1, c = v[i][j];
    const bool gsite = xo != yo;
    const unsigned g = gsite ? c : cross;
    const unsigned r = gsite ? (yo ? vv : hh) : (yo ? diag : c);
    const unsigned b = gsite ? (yo ? hh : vv) : (yo ? c : diag);
    return b | (g << 8) | (r << 16);
}

// The Bayer form of resize_u8c3_kernel's row loop: frames of sh * sw bytes at a uniform stride, the uniform row / column
// tables (xtab's byte offsets are 3 * source column), resize_combine and the same stores.  A row's taps y0 and
// y1 (= y0 or y0 + 1) are clamped to [1, sh - 2], a lane's x0 and x1 = min(x0 + 1, sw - 1) to [1, sw - 2]; the four
// sites (y0 | y1) x (x0 | x1) then lie in one 4x4 grid of raw bytes (rows y0 - 1 .. y0 + 1 and y1 + 1, columns x0 - 1 ..
// x0 + 1 and x1 + 1), loaded once and demosaiced into the 6-byte tap windows of the BGR kernel.
// Bounds: with sh, sw >= 3 the clamps keep every row in [0, sh - 1] and every column in [0, sw - 1], so every byte read
// lies inside its own frame, and frames are those of this launch: nothing is read before src or at or past
// src + n * sh * sw.  In the chunked host path that is the end of the chunk's landed bytes.  Loads are bytes, so there is
// no aligned word that could straddle the end and no clamped-row variant.
// The pattern is compile-time (FMT - RS_BAYER_RGGB = column flip | row flip << 1): the site parities fold into constants.
// LAYOUT: the frames are pitched as *lay says (the same grid of rows at other addresses).
template <bool WORD_STORE, int FMT, bool LAYOUT>
__device__ __forceinline__ void resize_bayer_rows(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, const int2 *__restrict__ xtab,
                                                  const int4 *__restrict__ ytab, unsigned row, unsigned row_end, int sh, int sw, int dh, int dw, int lane,
                                                  const ResizeLayout *__restrict__ lay)
{
    constexpr unsigned PX = (FMT - RS_BAYER_RGGB) & 1, PY = (FMT - RS_BAYER_RGGB) >> 1;
    const int p = (4 * lane) / 3;
    const unsigned rsh = 8u * (unsigned)(4 * lane - 3 * p);
    ResizeLayout L{};
    if constexpr (LAYOUT) L = *lay;
    const size_t frame_bytes = LAYOUT ? (size_t)L.stride : (size_t)sh * sw;
    const unsigned ymax = (unsigned)sh - 2u, xmax = (unsigned)sw - 2u;
    unsigned dy = row % (unsigned)dh;
    const uint8_t *frame = src + (size_t)(row / (unsigned)dh) * frame_bytes;
    uint8_t *drow = dst + (size_t)row * dw * 3;
    for (; row < row_end; ++row) {
        const int4 yt = __ldg(ytab + dy);
        const unsigned y0 = min(max((unsigned)yt.x, 1u), ymax), y1 = min(max((unsigned)yt.y, 1u), ymax);
        const uint8_t *rows[4];                                      // warp-uniform
        if constexpr (LAYOUT) {
            rows[0] = frame + (L.off[0] + (y0 - 1u) * L.pitch[0]); rows[1] = rows[0] + L.pitch[0]; rows[2] = rows[1] + L.pitch[0];
            rows[3] = frame + (L.off[0] + (y1 + 1u) * L.pitch[0]);
        } else {
            rows[0] = frame + (size_t)(y0 - 1u) * sw; rows[1] = rows[0] + sw; rows[2] = rows[1] + sw;
            rows[3] = frame + (size_t)(y1 + 1u) * sw;
        }
        const bool ystep = y1 != y0;
        const unsigned yo = (y0 ^ PY) & 1u;
        for (int dx0 = 0; dx0 < dw; dx0 += 32) {
            const int dx = dx0 + lane;
            const bool live = dx < dw;
            unsigned v = 0;
            if (live) {
                const int2 xt = __ldg(xtab + dx);
                const unsigned xa = (unsigned)xt.x / 3u;
                const unsigned x0 = min(max(xa, 1u), xmax), x1 = min(max(min(xa + 1u, (unsigned)sw - 1u), 1u), xmax);
                const bool xstep = x1 != x0;
                unsigned g[4][4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
#pragma unroll
                    for (int j = 0; j < 3; ++j) g[i][j] = __ldg(rows[i] + x0 - 1u + j);
                    g[i][3] = __ldg(rows[i] + x1 + 1u);
                }
                const unsigned xo = (x0 ^ PX) & 1u;
                const unsigned s00 = bayer_site(g, 0, 0, xo, yo), s01 = bayer_site(g, 0, 1, xo ^ 1u, yo);
                const unsigned s10 = bayer_site(g, 1, 0, xo, yo ^ 1u), s11 = bayer_site(g, 1, 1, xo ^ 1u, yo ^ 1u);
                const unsigned t00 = s00, t01 = xstep ? s01 : s00;
                const unsigned t10 = ystep ? s10 : t00, t11 = ystep ? (xstep ? s11 : s10) : t01;
                v = resize_combine(t00 | (t01 << 24), t01 >> 8, t10 | (t11 << 24), t11 >> 8, (unsigned)xt.y, (unsigned)yt.z, (unsigned)yt.w);
            }
            resize_store<WORD_STORE>(v, live, dx0, dx, dw, drow, lane, p, rsh);
        }
        drow += (size_t)dw * 3;
        if (++dy == (unsigned)dh) { dy = 0; frame += frame_bytes; }
    }
}

// ---- RGB, RGBA, BGRA, gray and planar RGB sources: cv2.cvtColor(COLOR_RGB2BGR / _RGBA2BGR / _BGRA2BGR / _GRAY2BGR) ------
// Each conversion selects (or, for gray, replicates) channels per pixel, and the resize treats the channels alike, so
// resize(convert(f)) = convert(resize(f)): the kernel resizes the source's own channels and writes them in B, G, R order.
// Packed RGB is the BGR row loop with the channel order swapped in resize_combine.  The others use resize_pix_rows.
// The RGBA / BGRA loops read one aligned 32-bit word per tap pixel when src is 4-byte aligned (frames are 4 * sh * sw
// bytes, so every frame and row then is); resize_u8c3 sends other sources to these byte-load variants of the two formats:
enum { RS_RGBA_BYTES = 13, RS_BGRA_BYTES = 14 };

// The horizontal and vertical pass of one channel: p0 / p1 = tap 0 | tap 1 << 8 of the two source rows (resize_combine).
__device__ __forceinline__ unsigned resize_channel(unsigned p0, unsigned p1, unsigned a01, unsigned B0, unsigned B1)
{
    return (__umulhi(B0, __dp2a_lo(a01, p0, 0u) >> 4) + __umulhi(B1, __dp2a_lo(a01, p1, 0u) >> 4) + 2u) >> 2;
}

// bytes 0..2 (the colour channels) of pixel x of a 4-byte-per-pixel row, as one word
__device__ __forceinline__ unsigned rgba_bytes(const uint8_t *row, unsigned x)
{
    const uint8_t *q = row + 4u * x;
    return (unsigned)__ldg(q) | ((unsigned)__ldg(q + 1) << 8) | ((unsigned)__ldg(q + 2) << 16);
}

// The gray / RGBA / BGRA / planar RGB form of resize_u8c3_kernel's row loop: frames of BPP * sh * sw bytes at a uniform
// stride, the uniform row / column tables (xtab's byte offsets are 3 * source column), the same stores.  Per source row
// and lane, the two tap pixels x0 and x1 = min(x0 + 1, sw - 1) (tap 1 has weight 0 where x0 = sw - 1):
//   GRAY:          two bytes, one channel resized and replicated into B, G and R (a third of the arithmetic);
//   RGBA / BGRA:   two aligned words (or, in the byte variants, the three colour bytes of each), resize_combine;
//   RGB_PLANAR:    two bytes from each of the three planes, whose row pointers are warp-uniform.
// Bounds: a source row index comes from ytab (clamped to [0, sh - 1]) and a column from xtab (in [0, sw - 1]) or its
// clamped successor, so every byte read (a word: the pixel's own four bytes) lies inside its own frame, and frames are
// those of this launch: nothing is read before src or at or past src + n * frame_bytes.  In the chunked host path that is
// the end of the chunk's landed bytes.  So there is no clamped-row variant.
// LAYOUT: the frames are pitched as *lay says; planar RGB then reads plane p's rows at off[p] + r * pitch[p], the others
// plane 0's.  The RGBA / BGRA word loads need every row 4-byte aligned: src, the stride and the pitch multiples of 4.
template <bool WORD_STORE, int FMT, bool LAYOUT>
__device__ __forceinline__ void resize_pix_rows(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, const int2 *__restrict__ xtab,
                                                const int4 *__restrict__ ytab, unsigned row, unsigned row_end, int sh, int sw, int dh, int dw, int lane,
                                                const ResizeLayout *__restrict__ lay)
{
    constexpr bool GRAY = FMT == RS_GRAY, PLANAR = FMT == RS_RGB_PLANAR;
    constexpr bool WORDS = FMT == RS_RGBA || FMT == RS_BGRA, RGB = FMT == RS_RGBA || FMT == RS_RGBA_BYTES;
    constexpr unsigned BPP = GRAY ? 1 : PLANAR ? 3 : 4;           // frame bytes per pixel
    constexpr unsigned ROW = PLANAR ? 1 : BPP;                    // row bytes per pixel (of one plane)
    const int p = (4 * lane) / 3;
    const unsigned rsh = 8u * (unsigned)(4 * lane - 3 * p);
    const size_t plane = (size_t)sh * sw;
    ResizeLayout L{};
    if constexpr (LAYOUT) L = *lay;
    const size_t frame_bytes = LAYOUT ? (size_t)L.stride : BPP * plane;
    unsigned dy = row % (unsigned)dh;
    const uint8_t *frame = src + (size_t)(row / (unsigned)dh) * frame_bytes;
    uint8_t *drow = dst + (size_t)row * dw * 3;
    for (; row < row_end; ++row) {
        const int4 yt = __ldg(ytab + dy);
        const uint8_t *r0, *r1;                                      // warp-uniform
        if constexpr (LAYOUT) {
            r0 = frame + (L.off[0] + (unsigned)yt.x * L.pitch[0]); r1 = frame + (L.off[0] + (unsigned)yt.y * L.pitch[0]);
        } else {
            r0 = frame + (size_t)yt.x * sw * ROW; r1 = frame + (size_t)yt.y * sw * ROW;
        }
        for (int dx0 = 0; dx0 < dw; dx0 += 32) {
            const int dx = dx0 + lane;
            const bool live = dx < dw;
            unsigned v = 0;
            if (live) {
                const int2 xt = __ldg(xtab + dx);
                const unsigned x0 = (unsigned)xt.x / 3u, x1 = min(x0 + 1u, (unsigned)sw - 1u);
                const unsigned a01 = (unsigned)xt.y, B0 = (unsigned)yt.z, B1 = (unsigned)yt.w;
                if constexpr (GRAY) {
                    v = 0x010101u * resize_channel(__ldg(r0 + x0) | ((unsigned)__ldg(r0 + x1) << 8),
                                                   __ldg(r1 + x0) | ((unsigned)__ldg(r1 + x1) << 8), a01, B0, B1);
                } else if constexpr (PLANAR) {
#pragma unroll
                    for (int ch = 0; ch < 3; ++ch) {                  // output B, G, R = planes 2, 1, 0
                        const uint8_t *q0 = r0 + (2 - ch) * plane, *q1 = r1 + (2 - ch) * plane;
                        if constexpr (LAYOUT) {
                            q0 = frame + (L.off[2 - ch] + (unsigned)yt.x * L.pitch[2 - ch]);
                            q1 = frame + (L.off[2 - ch] + (unsigned)yt.y * L.pitch[2 - ch]);
                        }
                        v |= resize_channel(__ldg(q0 + x0) | ((unsigned)__ldg(q0 + x1) << 8),
                                            __ldg(q1 + x0) | ((unsigned)__ldg(q1 + x1) << 8), a01, B0, B1) << (8 * ch);
                    }
                } else if constexpr (WORDS) {
                    const unsigned *w0 = reinterpret_cast<const unsigned *>(r0), *w1 = reinterpret_cast<const unsigned *>(r1);
                    v = resize_combine<RGB, 4>(__ldg(w0 + x0), __ldg(w0 + x1), __ldg(w1 + x0), __ldg(w1 + x1), a01, B0, B1);
                } else {
                    v = resize_combine<RGB, 4>(rgba_bytes(r0, x0), rgba_bytes(r0, x1), rgba_bytes(r1, x0), rgba_bytes(r1, x1), a01, B0, B1);
                }
            }
            resize_store<WORD_STORE>(v, live, dx0, dx, dw, drow, lane, p, rsh);
        }
        drow += (size_t)dw * 3;
        if (++dy == (unsigned)dh) { dy = 0; frame += frame_bytes; }
    }
}

constexpr bool rs_is_yuv(int fmt) { return fmt == RS_YUV_NV12 || fmt == RS_YUV_I420 || fmt == RS_YUV_YUYV; }
constexpr bool rs_is_bayer(int fmt) { return fmt >= RS_BAYER_RGGB && fmt <= RS_BAYER_BGGR; }
constexpr bool rs_is_pix_rows(int fmt)          // the formats of resize_pix_rows
{
    return fmt == RS_GRAY || fmt == RS_RGB_PLANAR || fmt == RS_RGBA || fmt == RS_BGRA || fmt == RS_RGBA_BYTES || fmt == RS_BGRA_BYTES;
}

// resident CTAs of 256 threads per SM the launch plans for (= the kernel's __launch_bounds__): 6 at 40 registers; the
// ragged descriptor bookkeeping needs 48 (5 CTAs) and the 4:2:0 instantiations, which keep luma and chroma row pointers of
// both source rows, up to 64 (4 CTAs) to run without spills; YUYV fits 40; the Bayer instantiations, which keep a lane's
// 4x4 grid of raw bytes and four row pointers, need up to 64 (4 CTAs); gray and the RGBA / BGRA word loads fit 40; RGB
// (the BGR loop with its word stores), the RGBA / BGRA byte loads and planar RGB need up to 48 (5 CTAs)
// The pitched (LAYOUT) instantiations keep a frame stride and plane offsets / pitches besides: gray still fits 40, the
// packed 3-byte loops, YUYV and RGBA / BGRA (both load variants) need up to 48 (5 CTAs), 4:2:0, Bayer and planar RGB up to
// 64 (4 CTAs) to run without spills
constexpr int resize_ctas_per_sm(bool ragged, int fmt, bool layout = false)
{
    if (layout) return fmt == RS_YUV_NV12 || fmt == RS_YUV_I420 || rs_is_bayer(fmt) || fmt == RS_RGB_PLANAR ? 4 : fmt == RS_GRAY ? 6 : 5;
    return ragged ? 5 : fmt == RS_YUV_NV12 || fmt == RS_YUV_I420 || rs_is_bayer(fmt) ? 4
         : fmt == RS_RGB || fmt == RS_RGB_PLANAR || fmt == RS_RGBA_BYTES || fmt == RS_BGRA_BYTES ? 5 : 6;
}

// One WARP = a contiguous run of output rows of the batch (so the row bookkeeping is incremental: no divisions), one
// whole row at a time, chunk after chunk: the ~70 instructions of row bookkeeping are paid once per row, not once per
// 32-pixel chunk (with one CTA per row every warp repeated them for its single chunk: 150 instead of 85 instructions per
// chunk).  Everything that depends on the row only (taps, weights, row pointers, their misalignment) is warp-uniform.
// WORD_STORE needs dst 4-byte aligned and dw % 4 == 0, so that every row and every 32-pixel chunk starts on a word.
// RAGGED: the frames have different source sizes (every frame still becomes dh x dw).  Frame f is described by
// frames[f] = {byte offset in src, row pitch, geometry g}; its row / column tables are ytab + g * dh / xtab + g * dw.  The
// descriptor is loaded when dy wraps, so its cost is warp-uniform and paid once per frame.  Otherwise frames are
// sh x sw and packed at a uniform stride.
// FMT: the source format, RS_BGR (uint8 [sh][sw][3]), RS_RGB (the same loop with R and B swapped; uniform stride only),
// one of the YUV layouts (uniform stride only; resize_yuv_rows), one of the Bayer patterns (uniform stride only;
// resize_bayer_rows) or gray, RGBA / BGRA (either load variant) and planar RGB (uniform stride only; resize_pix_rows).
// LAYOUT (not RAGGED): the frames are sh x sw at the pitched layout `frames` points to (a ResizeLayout: no new kernel
// argument), src = the first byte of frame 0's planes and src_bytes the bytes from there to the end of the launch's last
// row.  The packed 3-byte loop then takes its frame stride and row pitch from the record, and the rule "rows whose
// window could reach past the end" holds as it is: a window reaches at most 11 bytes past its pixel, so less than
// pitch + 12 past its row's start, whatever the pitch.  Bytes between rows (padding) are read only as tap 1 of a
// right-border pixel or the slack of a word, both with weight 0; rows that start in the first word of the buffer take the
// clamped byte loads too, so nothing before src is read.
template <bool WORD_STORE, bool RAGGED, int FMT = RS_BGR, bool LAYOUT = false>
__global__ void __launch_bounds__(256, resize_ctas_per_sm(RAGGED, FMT, LAYOUT)) resize_u8c3_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
                                                          const int2 *__restrict__ xtab, const int4 *__restrict__ ytab,
                                                          const ResizeFrame *__restrict__ frames,
                                                          unsigned rows, unsigned rows_per_warp, int sh, int sw, int dh, int dw, size_t src_bytes)
{
    const int lane = threadIdx.x & 31;
    unsigned row = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * rows_per_warp;
    if (row >= rows) return;
    const unsigned row_end = min(rows, row + rows_per_warp);
    static_assert(!(RAGGED && LAYOUT), "a pitched launch is one size");
    const ResizeLayout *lay = reinterpret_cast<const ResizeLayout *>(frames);
    if constexpr (rs_is_bayer(FMT)) {
        static_assert(!RAGGED, "Bayer sources are one size per launch");
        resize_bayer_rows<WORD_STORE, FMT, LAYOUT>(src, dst, xtab, ytab, row, row_end, sh, sw, dh, dw, lane, lay);
        return;
    } else if constexpr (rs_is_pix_rows(FMT)) {
        static_assert(!RAGGED, "gray, RGBA, BGRA and planar sources are one size per launch");
        resize_pix_rows<WORD_STORE, FMT, LAYOUT>(src, dst, xtab, ytab, row, row_end, sh, sw, dh, dw, lane, lay);
        return;
    } else if constexpr (rs_is_yuv(FMT)) {
        static_assert(!RAGGED, "YUV sources are one size per launch");
        resize_yuv_rows<WORD_STORE, FMT, LAYOUT>(src, dst, xtab, ytab, row, row_end, sh, sw, dh, dw, lane, lay);
        return;
    } else {
        static_assert(FMT == RS_BGR || (FMT == RS_RGB && !RAGGED), "the packed 3-byte row loop takes BGR, and RGB at a uniform stride");
    }
    const size_t delta = reinterpret_cast<uintptr_t>(src) & 3;                             // word-aligned view of the source
    const unsigned char *base = src - delta;
    const size_t end = delta + src_bytes;                                                  // one past the last source byte
    const int p = (4 * lane) / 3;
    const unsigned rsh = 8u * (unsigned)(4 * lane - 3 * p);
    unsigned dy = row % (unsigned)dh;
    size_t src_frame = 0, src_row, frame_off;
    unsigned f = row / (unsigned)dh, geom = 0;
    auto load_frame = [&](unsigned fi) {
        const int4 d = __ldg(reinterpret_cast<const int4 *>(frames) + fi);
        frame_off = delta + ((size_t)(unsigned)d.x | ((size_t)(unsigned)d.y << 32));
        src_row = (unsigned)d.z;
        geom = (unsigned)d.w;
    };
    if constexpr (RAGGED) {
        load_frame(f);
    } else if constexpr (LAYOUT) {
        src_frame = lay->stride; src_row = lay->pitch[0];
        frame_off = delta + lay->off[0] + (size_t)f * src_frame;
    } else {
        src_frame = (size_t)sh * sw * 3; src_row = (size_t)sw * 3;
        frame_off = delta + (size_t)f * src_frame;
    }
    uint8_t *drow = dst + (size_t)row * dw * 3;
    for (; row < row_end; ++row) {
        const int4 yt = __ldg(ytab + (RAGGED ? geom * (unsigned)dh + dy : dy));
        const size_t o0 = frame_off + (size_t)yt.x * src_row, o1 = frame_off + (size_t)yt.y * src_row;
        const unsigned char *r0 = base + (o0 & ~(size_t)3), *r1 = base + (o1 & ~(size_t)3);
        const unsigned d0 = (unsigned)o0 & 3u, d1 = (unsigned)o1 & 3u;
        // a window reaches at most 11 bytes past the start of its pixel; rows for which that stays inside the buffer need no
        // clamp (in a ragged batch, bytes past a frame's last pixel belong to the next frame and carry zero weight)
        // LAYOUT: nor the rows that start in the buffer's first word (o0 < 4, o0 <= o1), whose first aligned word would
        // hold bytes before src: src is the first byte of the span, and a pitched call reads nothing outside its span
        const size_t omax = o0 > o1 ? o0 : o1;
        if (omax + src_row + 12 <= end && (!LAYOUT || o0 >= 4)) {
            resize_one_row<WORD_STORE, false, FMT == RS_RGB, LAYOUT>(r0, r1, d0, d1, 0u, 0u, (unsigned)yt.z, (unsigned)yt.w, RAGGED ? xtab + geom * (unsigned)dw : xtab, drow, dw, lane, 0, 1, p, rsh);
        } else {
            const size_t room0 = end - 1 - (o0 & ~(size_t)3), room1 = end - 1 - (o1 & ~(size_t)3);
            resize_one_row<WORD_STORE, true, FMT == RS_RGB>(r0, r1, d0, d1, (unsigned)room0, (unsigned)room1, (unsigned)yt.z, (unsigned)yt.w, RAGGED ? xtab + geom * (unsigned)dw : xtab, drow, dw, lane, 0, 1, p, rsh);
        }
        drow += (size_t)dw * 3;
        if (++dy == (unsigned)dh) {
            dy = 0;
            if constexpr (RAGGED) { if (row + 1 < row_end) load_frame(++f); }
            else frame_off += src_frame;
        }
    }
}

// one wave of resident CTAs (8 warps each), equal runs of rows per warp
template <bool RAGGED, int FMT = RS_BGR, bool LAYOUT = false>
static cudaError_t resize_launch(const uint8_t *src, size_t src_bytes, const ResizeFrame *frames, int n, int sh, int sw, uint8_t *dst,
                                 int dh, int dw, const int2 *xtab_dev, const int4 *ytab_dev, int sm_count, cudaStream_t st)
{
    if (n <= 0) return cudaSuccess;
    const size_t rows = (size_t)n * dh;
    if (rows > 0x7fffffffull) return cudaErrorInvalidValue;
    const int threads = 256;
    const size_t max_warps = (size_t)(sm_count > 0 ? sm_count : 148) * resize_ctas_per_sm(RAGGED, FMT, LAYOUT) * (threads / 32);
    const unsigned rows_per_warp = (unsigned)((rows + max_warps - 1) / max_warps);
    const size_t warps = (rows + rows_per_warp - 1) / rows_per_warp;
    const size_t blocks = (warps + threads / 32 - 1) / (threads / 32);
    if ((reinterpret_cast<uintptr_t>(dst) & 3) == 0 && dw % 4 == 0)
        resize_u8c3_kernel<true, RAGGED, FMT, LAYOUT><<<(unsigned)blocks, threads, 0, st>>>(src, dst, xtab_dev, ytab_dev, frames, (unsigned)rows, rows_per_warp, sh, sw, dh, dw, src_bytes);
    else
        resize_u8c3_kernel<false, RAGGED, FMT, LAYOUT><<<(unsigned)blocks, threads, 0, st>>>(src, dst, xtab_dev, ytab_dev, frames, (unsigned)rows, rows_per_warp, sh, sw, dh, dw, src_bytes);
    return cudaGetLastError();
}

size_t camera_frame_bytes(int format, int sh, int sw)
{
    const size_t px = (size_t)sh * sw;
    switch (format) {
    case RS_YUV_NV12: case RS_YUV_I420: return px + px / 2;
    case RS_YUV_YUYV: return 2 * px;
    case RS_BAYER_RGGB: case RS_BAYER_GRBG: case RS_BAYER_GBRG: case RS_BAYER_BGGR: case RS_GRAY: return px;
    case RS_BGR: case RS_RGB: case RS_RGB_PLANAR: return 3 * px;
    case RS_RGBA: case RS_BGRA: return 4 * px;
    default: return 0;
    }
}

int source_planes(int format, int sh, int sw, int rows[3], int row_bytes[3])
{
    auto set = [&](int p, int r, int b) { rows[p] = r; row_bytes[p] = b; };
    switch (format) {
    case RS_YUV_NV12: set(0, sh, sw); set(1, sh / 2, sw); return 2;
    case RS_YUV_I420: set(0, sh, sw); set(1, sh / 2, sw / 2); set(2, sh / 2, sw / 2); return 3;
    case RS_YUV_YUYV: set(0, sh, 2 * sw); return 1;
    case RS_BAYER_RGGB: case RS_BAYER_GRBG: case RS_BAYER_GBRG: case RS_BAYER_BGGR: case RS_GRAY: set(0, sh, sw); return 1;
    case RS_BGR: case RS_RGB: set(0, sh, 3 * sw); return 1;
    case RS_RGBA: case RS_BGRA: set(0, sh, 4 * sw); return 1;
    case RS_RGB_PLANAR: set(0, sh, sw); set(1, sh, sw); set(2, sh, sw); return 3;
    default: return 0;
    }
}

// The launches of the pitched layout: the uniform dispatch below with LAYOUT set and the record as `frames`
static cudaError_t resize_u8c3_pitched(const uint8_t *src, size_t src_bytes, int fmt, const ResizeLayout *lay, bool word_pitch, int n, int sh, int sw,
                                       uint8_t *dst, int dh, int dw, const int2 *xtab_dev, const int4 *ytab_dev, int sm_count, cudaStream_t st)
{
    const ResizeFrame *f = reinterpret_cast<const ResizeFrame *>(lay);
#define RS_PITCHED(F) resize_launch<false, F, true>(src, src_bytes, f, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st)
    switch (fmt) {
    case RS_BGR:        return RS_PITCHED(RS_BGR);
    case RS_YUV_NV12:   return RS_PITCHED(RS_YUV_NV12);
    case RS_YUV_I420:   return RS_PITCHED(RS_YUV_I420);
    case RS_YUV_YUYV:   return RS_PITCHED(RS_YUV_YUYV);
    case RS_BAYER_RGGB: return RS_PITCHED(RS_BAYER_RGGB);
    case RS_BAYER_GRBG: return RS_PITCHED(RS_BAYER_GRBG);
    case RS_BAYER_GBRG: return RS_PITCHED(RS_BAYER_GBRG);
    case RS_BAYER_BGGR: return RS_PITCHED(RS_BAYER_BGGR);
    case RS_RGB:        return RS_PITCHED(RS_RGB);
    case RS_GRAY:       return RS_PITCHED(RS_GRAY);
    case RS_RGB_PLANAR: return RS_PITCHED(RS_RGB_PLANAR);
    case RS_RGBA: case RS_BGRA: {
        const bool words = word_pitch && (reinterpret_cast<uintptr_t>(src) & 3) == 0;     // every row 4-byte aligned
        if (fmt == RS_RGBA) return words ? RS_PITCHED(RS_RGBA) : RS_PITCHED(RS_RGBA_BYTES);
        return words ? RS_PITCHED(RS_BGRA) : RS_PITCHED(RS_BGRA_BYTES);
    }
    default:            return cudaErrorInvalidValue;
    }
#undef RS_PITCHED
}

cudaError_t resize_u8c3(const uint8_t *src, size_t src_bytes, int fmt, const ResizeFrame *frames_dev, int n, int sh, int sw,
                        uint8_t *dst, int dh, int dw, const int2 *xtab_dev, const int4 *ytab_dev, int sm_count, cudaStream_t st,
                        const ResizeLayout *layout_dev, bool word_pitch)
{
    if (layout_dev)
        return frames_dev ? cudaErrorInvalidValue
                          : resize_u8c3_pitched(src, src_bytes, fmt, layout_dev, word_pitch, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    if (frames_dev)
        return fmt == RS_BGR ? resize_launch<true>(src, src_bytes, frames_dev, n, 0, 0, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st) : cudaErrorInvalidValue;
    switch (fmt) {
    case RS_BGR:      return resize_launch<false>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    case RS_YUV_NV12: return resize_launch<false, RS_YUV_NV12>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    case RS_YUV_I420: return resize_launch<false, RS_YUV_I420>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    case RS_YUV_YUYV: return resize_launch<false, RS_YUV_YUYV>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    case RS_BAYER_RGGB: return resize_launch<false, RS_BAYER_RGGB>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    case RS_BAYER_GRBG: return resize_launch<false, RS_BAYER_GRBG>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    case RS_BAYER_GBRG: return resize_launch<false, RS_BAYER_GBRG>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    case RS_BAYER_BGGR: return resize_launch<false, RS_BAYER_BGGR>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    case RS_RGB:        return resize_launch<false, RS_RGB>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    case RS_GRAY:       return resize_launch<false, RS_GRAY>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    case RS_RGB_PLANAR: return resize_launch<false, RS_RGB_PLANAR>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    case RS_RGBA: case RS_BGRA: {
        const bool words = (reinterpret_cast<uintptr_t>(src) & 3) == 0;
        if (fmt == RS_RGBA)
            return words ? resize_launch<false, RS_RGBA>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st)
                         : resize_launch<false, RS_RGBA_BYTES>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
        return words ? resize_launch<false, RS_BGRA>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st)
                     : resize_launch<false, RS_BGRA_BYTES>(src, src_bytes, nullptr, n, sh, sw, dst, dh, dw, xtab_dev, ytab_dev, sm_count, st);
    }
    default:          return cudaErrorInvalidValue;
    }
}

void resize_geometry_tables(int sh, int sw, int dh, int dw, int4 *ytab, int2 *xtab)
{
    resize_axis_table(sh, dh, false, 1, ytab);               // row taps; weights pre-shifted for the kernel's high multiply
    for (int d = 0; d < dh; ++d) { ytab[d].z <<= 16; ytab[d].w <<= 16; }
    std::vector<int4> t((size_t)dw);
    resize_axis_table(sw, dw, true, 3, t.data());            // column taps as byte offsets inside a row; tap 1 = the next pixel
    for (int d = 0; d < dw; ++d) xtab[d] = make_int2(t[d].x, t[d].z | (t[d].w << 16));
}

}  // namespace yb
