// conv_fs.cu — the first layer on tcgen05 ("first layer, slots"): 3x3 / pad 1 convolution of the 3-channel camera frame to 16
// channels + requantisation + leaky-ReLU + 2x2 max-pool, for the geometries the benchmark runs (pooled width >= 128).
//
// Replaces first_conv (c_embedding/yolo_forward.c:269-418) and conv1 + tracker + pool (models/slim_yolo_v2.py:220-231), like
// conv_first.cu, which stays the general kernel (un-pooled / wide / narrow / BGR-byte first layers).  conv_first.cu runs on
// warp-level integer MMAs and is bound by instruction issue (61 % of the issue slots, 0.22 ms per 256 frames of 416x416 against
// 0.04 ms of HBM time).  Here the convolution runs on tcgen05 without an im2col row per output pixel:
//
//   * K.  A pixel is one 32-bit word (R, G, B, 0).  A SLOT is 16 bytes = the words of pixels 2j-1, 2j, 2j+1, 2j+2 of one input row.
//     Output pixel x = 2j reads its three horizontal taps from words 0-2 of slot j, output pixel x = 2j+1 from words 1-3: ONE slot
//     array serves both x parities, the parity only selects which three of the four weight words are non-zero.  The GEMM N dimension
//     carries two x parities x two output rows x 16 channels (column e * 32 + dy * 16 + co = channel co of pixel (2Y + dy, 2j + e)),
//     so K spans the four input rows 2Y-1 .. 2Y+2 = four slots = two K = 32 instructions of N = 64; the weight images hold zeros
//     where kh = row - dy or kw = word - e falls outside 0..2.  All four members of pooled pixel (Y, j) land in ONE TMEM lane: the
//     2x2 max-pool is three integer maxima per channel, no shuffles (requantisation is monotone: slim_yolo_v2.py:229-231).
//   * rows.  Input rows 2i-1 ("odd") and 2i ("even") form PAIR-ROW i; odd and even rows live in two arrays with the same pitch of
//     OW slots.  Pooled row Y reads pair-rows Y and Y+1; within one instruction the second K chunk (the even row) is the first
//     one's address + LBO = the distance between the two arrays.  Because the pitch is exactly OW slots, the 128 M rows of an
//     instruction may run over the end of a row into the next pair-row: a tile is ANY 128 consecutive pooled pixels of the frame
//     in raster order (416x416: 43264 = 338 x 128, no ragged tiles), and the output of a tile is 2 KB of consecutive bytes.
//   * the arrays are rings of R pair-rows (+ a mirror of the first row behind the last one, so that a tile that starts in the
//     last ring row continues into valid data).  Builder warps fill them: the raw frame rows arrive in a ring of 16 pair-rows by
//     1-D bulk copies (no register staging, no exposed HBM latency), a builder lane reads two pixels, quantises them through the
//     4096-entry table (camera_to_inpBuf + pixel_norm_quantize, yolo_forward.c:57-123), takes one word from each neighbour by
//     shuffles and writes the slot with one conflict-free 128-bit store: 8 bytes of shared-memory writes per pixel, where an
//     im2col row per pixel would need 32 and byte shuffling.
//
// Shared-memory port budget per 512 input pixels (one tile): 4 KB of slot writes + 2 x (4 KB of A + 2 KB of B) operand reads.
// What bounds the kernel is instruction issue (~1300 warp instructions per tile: 4 x 210 in the requantisation epilogue, ~310 in
// the builders, ~130 in the issuer; ~3 issued per clock and SM), see profiles/README.md.
//
// Warp roles (928 threads): warps 0-3 MMA issuers (tile t -> issuer t % 4), warp 4 raw-row loader (one lane), warps 5-12 slot
// builders (teams of two warps, one input row each; four pair-rows in flight), warps 13-28 four epilogue groups (tile t -> group
// t % 4; one warp per TMEM lane quarter).  Tile t uses TMEM buffer t % 8 (64 columns; t % 4 and 128 columns for 32 channels).
#include "kernels.h"
#include "ptx.cuh"
#include "epilogue.cuh"
#include <cstdio>
#include <cstdlib>
#include <time.h>

namespace yb {

// YB_FS_TIMELINE builds (tools/dbg_build.sh): clock64 stamps of CTA 0, 24 slots per entry: builder warps 0 and 7 (slots 0-5 / 6-11: start, raw row
// there, ring slot free, stored, fenced, published), issuer 0 (12-15: loop top, rows there, accumulator free, issued), epilogue group 0 (16-17)
#ifdef YB_FS_TIMELINE
#define FS_STAMP(n, slot) do { if (p.dbg && blockIdx.x == 0 && (n) < 64 && lane == 0) p.dbg[(n) * 24 + (slot)] = clock64(); } while (0)
#else
#define FS_STAMP(n, slot) do { } while (0)
#endif
// YB_FS_WATCH builds: every role publishes its progress to host-mapped memory; the launcher prints the table if the kernel does not finish
#ifdef YB_FS_WATCH
#define FS_WATCH(slot, val) do { if (p.watch && lane == 0) ((volatile unsigned *)p.watch)[blockIdx.x * 32 + (slot)] = (unsigned)(val); } while (0)
#else
#define FS_WATCH(slot, val) do { } while (0)
#endif
#define FS_STAMP_B(slot) do { if (bw == 0) FS_STAMP(gl_row / FS_NTEAM, slot); else if (bw == 7) FS_STAMP(gl_row / FS_NTEAM, 6 + (slot)); } while (0)

constexpr int FS_THREADS = 928;
constexpr int FS_NI = 4;                 // MMA issuer warps 0-3 (tile t -> issuer t % 4): a lone warp needs ~1250 cycles per tile (barrier polls, descriptor
                                         // arithmetic, MMAs, commits: one dependent instruction every ~8 cycles next to the other warps)
constexpr int FS_LW = 4;                 // raw-row loader warp
constexpr int FS_BW0 = 5, FS_NBW = 8;    // builder warps 5 .. 12: teams of two (odd input row / even input row); team m fills the pair-rows m, m + 4, ...
constexpr int FS_NTEAM = FS_NBW / 2;
constexpr int FS_EW0 = 13, FS_EG = 4;    // epilogue warps 13 .. 28: four groups of four (any four consecutive warps cover the four TMEM lane quarters)
constexpr int FS_RAWR = 16;              // raw pair-row ring: the loader runs up to 16 pair-rows ahead of the builders (HBM latency)
constexpr int FS_RMAX = 16;              // slot ring rows (barrier space)
// CO output channels (16: slim_yolo_v2, 32: darknet19): a tile's accumulators are 4 CO TMEM columns (x parity, row, channel)
constexpr int FS_TBUF_MAX = 8;
constexpr int FS_SEGW = 30;              // pixel pairs a builder warp produces per pass (lanes 0 and 31 only feed their neighbours)

struct FsParams {
    const void *src;             // SRC 1: uint16 RGB444 frames [n][H][W]; SRC 0: int8 NHWC4 [n][H][W][4]; SRC 2: uint8 BGR images [n][H][W][3]
    const int *lut;              // SRC 1: 4096 packed (R,G,B,0) words; SRC 2: three 256-byte tables (R from byte 2, G, B: quantize.cu)
    int n_img, H, W, OH, OW;
    int ohw;                     // OH * OW pooled pixels per frame
    int upi;                     // units (tiles of 128 pooled pixels) per frame
    int total_units;
    unsigned ow_magic, upi_magic;    // ceil(2^32 / OW), ceil(2^32 / upi)
    int R, MR;                   // ring rows, mirrored rows
    int segs;                    // builder passes per input row = ceil(OW / 30)
    uint32_t row_bytes;          // one raw input row
    uint32_t arr_bytes;          // one slot array: (R + MR) * OW * 16, rounded up to 128
    uint32_t off_lut, off_raw, off_bias, off_bar, off_arr;
    int xsplit;
    int co;                      // 16 or 32 output channels = bytes per output pixel
    const int8_t *wgt;           // [cout_pad][9][4]
    const int *bias_sh;
    LayerQ q;
    EpiConst k;
    int8_t *out;
    unsigned *ovf;
    long long *dbg;
    unsigned *watch;
};

// mbarrier wait with a suspend-time hint: the warp sleeps in hardware until the phase completes (or the hint expires) instead of
// re-issuing the poll every few hundred cycles (the epilogue groups wait ~60 % of the time: ~35 polls per tile without it)
__device__ __forceinline__ void mbar_wait_hint(uint32_t bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(bar), "r"(parity), "r"(20000u) : "memory");
    } while (!done);
}

// predicated 128-bit shared store (a predicate, not a branch: the shuffles of the next pass are not held behind a reconvergence point)
__device__ __forceinline__ void st_shared_v4_if(bool pred, uint32_t addr, unsigned a, unsigned b, unsigned c, unsigned d)
{
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %5, 0;\n@p st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n}"
                 ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d), "r"((unsigned)pred) : "memory");
}

// The frames a CTA works on: global units [U0, U1) cut at frame boundaries.
struct FsSeg {
    int img, ua, ub;             // units [ua, ub) of frame img
    int ia, ib;                  // pair-rows ia .. ib feed them
};
__device__ __forceinline__ bool fs_next_seg(const FsParams &p, int &U, int U1, FsSeg &s)
{
    if (U >= U1) return false;
    s.img = p.upi == 1 ? U : (int)__umulhi((unsigned)U, p.upi_magic);
    s.ua = U - s.img * p.upi;
    s.ub = min(p.upi, s.ua + (U1 - U));
    U += s.ub - s.ua;
    const int qend = min(128 * s.ub, p.ohw);
    s.ia = (int)__umulhi((unsigned)(128 * s.ua), p.ow_magic);
    s.ib = min(p.OH, (int)__umulhi((unsigned)(qend - 1), p.ow_magic) + 1);
    return true;
}

// (Accumulators pre-biased with the fp32 magic constant by tcgen05.st from the epilogue warps, which would save the 16 int -> float
// conversions per thread and tile, were measured and rejected: re-arming 64 columns + tcgen05.wait::st costs ~1500 cycles per tile
// and group, 0.186 -> 0.260 ms.)
template <int EPI, bool ACT, int CO>
__device__ __forceinline__ void fs_epilogue_tile(const FsParams &p, const EpiPk &kp, uint32_t taddr, int q, int img, const int *s_bias, uint32_t bar_tempty, unsigned &ovf)
{
    const bool valid = q < p.ohw;
    int pos = q;
    if (CO == 16 && p.xsplit) {
        const int pr = (int)__umulhi((unsigned)q, p.ow_magic), j = q - pr * p.OW;
        pos = pr * p.OW + (j & 1) * (p.OW >> 1) + (j >> 1);
    }
    uint4 *dst = reinterpret_cast<uint4 *>(p.out + ((size_t)img * p.ohw + pos) * CO);
    unsigned w[4];
#pragma unroll
    for (int h = 0; h < CO / 8; ++h) {                         // channels 8h .. 8h + 7
        int a[8], b[8], c[8], d[8];
        tmem_ld8(taddr + 8 * h, a);                            // x even, row 2Y
        tmem_ld8(taddr + CO + 8 * h, b);                       // x even, row 2Y + 1
        tmem_ld8(taddr + 2 * CO + 8 * h, c);                   // x odd,  row 2Y
        tmem_ld8(taddr + 3 * CO + 8 * h, d);                   // x odd,  row 2Y + 1
        tmem_ld_wait();
        if (h == CO / 8 - 1) { tc_fence_before(); mbar_arrive(bar_tempty); }      // all of the tile's accumulators are in registers
#pragma unroll
        for (int j = 0; j < 8; ++j) a[j] = max(max(a[j], b[j]), max(c[j], d[j]));
        w[2 * (h & 1)] = requant4_pk<EPI, ACT>(&a[0], s_bias, 8 * h, p, kp, ovf, valid);
        w[2 * (h & 1) + 1] = requant4_pk<EPI, ACT>(&a[4], s_bias, 8 * h + 4, p, kp, ovf, valid);
        if ((h & 1) && valid) dst[h >> 1] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

template <int EPI, int SRC, int CO>
__global__ void __launch_bounds__(FS_THREADS, 1) conv3x3_fs_kernel(const FsParams p)
{
    // Accumulator columns per tile, TMEM buffers.  Tile t: issuer t % 4, epilogue group t % 4, buffer t % TBUF, use t / TBUF of that
    // buffer.  TBUF is a multiple of 4, so every buffer belongs to ONE issuer warp and ONE epilogue group: whoever waits for a phase
    // of `tfull` / `tempty` by parity took part in the previous phase itself, so an older phase can never satisfy the wait.  (With
    // three issuers over 4 / 8 buffers a stalled issuer let another one run two uses ahead of the drain: a deadlock at >= 64 tiles
    // per CTA with four buffers, found with the YB_FS_WATCH build.)
    constexpr int NCOL = 4 * CO, TBUF = 512 / NCOL;
    static_assert(TBUF % FS_NI == 0 && TBUF % FS_EG == 0, "buffers are owned");
    static_assert(CO == 16 || CO == 32, "16 or 32 output channels");
    pdl_launch_dependents();
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 127u) & ~127u;
    uint8_t *base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;     // broadcast: provably warp-uniform

    const uint32_t bsm = base;                                 // two weight images of NCOL x 32 bytes
    unsigned *s_lut = reinterpret_cast<unsigned *>(base_ptr + p.off_lut);
    const uint8_t *s_rawp = base_ptr + p.off_raw;
    const uint32_t raw0 = base + p.off_raw;
    int *s_bias = reinterpret_cast<int *>(base_ptr + p.off_bias);
    const uint32_t bar0 = base + p.off_bar;
    const uint32_t arr0 = base + p.off_arr;
    auto bar_rawfull = [&](int s) { return bar0 + 8u * s; };
    auto bar_rawempty = [&](int s) { return bar0 + 8u * (FS_RAWR + s); };
    auto bar_full = [&](int s) { return bar0 + 8u * (2 * FS_RAWR + s); };
    auto bar_empty = [&](int s) { return bar0 + 8u * (2 * FS_RAWR + FS_RMAX + s); };
    auto bar_tfull = [&](int b) { return bar0 + 8u * (2 * FS_RAWR + 2 * FS_RMAX + b); };
    auto bar_tempty = [&](int b) { return bar0 + 8u * (2 * FS_RAWR + 2 * FS_RMAX + FS_TBUF_MAX + b); };
    const uint32_t tmem_slot = bar0 + 8u * (2 * FS_RAWR + 2 * FS_RMAX + 2 * FS_TBUF_MAX);
    volatile uint32_t *tmem_slot_ptr = reinterpret_cast<volatile uint32_t *>(base_ptr + p.off_bar + 8u * (2 * FS_RAWR + 2 * FS_RMAX + 2 * FS_TBUF_MAX));
    const uint32_t raw_slot_bytes = 2u * p.row_bytes;

    if (threadIdx.x == 0) {
        for (int s = 0; s < FS_RAWR; ++s) { mbar_init(bar_rawfull(s), 1); mbar_init(bar_rawempty(s), 64); }
        for (int s = 0; s < FS_RMAX; ++s) { mbar_init(bar_full(s), 64); mbar_init(bar_empty(s), FS_NI); }
        for (int b = 0; b < TBUF; ++b) { mbar_init(bar_tfull(b), 1); mbar_init(bar_tempty(b), 128); }
        fence_barrier_init();
    }
    if (warp == 0) { __syncwarp(); tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
    // weight images: image bi = K chunks (2 bi, 2 bi + 1) = input rows (2Y - 1 + 2 bi, 2Y + 2 bi); GEMM column n = e * 2 CO + dy * CO + co =
    // channel co of output pixel (row 2Y + dy, x = 2j + e); word (n / 8, chunk, n % 8, w) of the no-swizzle K-major layout = the 4 channel
    // bytes of tap (kh = chunk row - dy, kw = w - e): the slot of pooled pixel j holds pixels 2j-1 .. 2j+2, an even x reads words 0-2, an odd x words 1-3
    for (int wd = threadIdx.x; wd < 16 * NCOL; wd += FS_THREADS) {
        const int bi = wd / (8 * NCOL), rem = wd - bi * (8 * NCOL);
        const int n = ((rem >> 6) << 3) | ((rem >> 2) & 7), cc = (rem >> 5) & 1, w = rem & 3;
        const int e = n / (2 * CO), dy = (n / CO) & 1, co = n % CO, kh = 2 * bi + cc - dy, kw = w - e;
        unsigned v = 0;
        if (kh >= 0 && kh <= 2 && kw >= 0 && kw <= 2) v = __ldg(reinterpret_cast<const unsigned *>(p.wgt) + co * 9 + kh * 3 + kw);
        reinterpret_cast<unsigned *>(base_ptr)[wd] = v;
    }
    if (SRC == 1) for (int i = threadIdx.x; i <= 4096; i += FS_THREADS) s_lut[i] = i < 4096 ? (unsigned)__ldg(p.lut + i) : 0u;   // entry 4096: outside the frame
    if (SRC == 2) for (int i = threadIdx.x; i < 192; i += FS_THREADS) s_lut[i] = (unsigned)__ldg(p.lut + i);
    if (threadIdx.x < CO) {
        const int b = p.bias_sh[threadIdx.x];
        s_bias[threadIdx.x] = (EPI == EPI_F_RNE || EPI == EPI_F_RNE_NOHI) ? __float_as_int((float)b) : b;
    }
    fence_proxy_async();                                       // the weight images are read by the tensor core (async proxy)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    pdl_wait();

    const int G = (int)gridDim.x;
    const int U0 = (int)(((long long)p.total_units * blockIdx.x) / G), U1 = (int)(((long long)p.total_units * (blockIdx.x + 1)) / G);
    const uint32_t row_pitch = (uint32_t)p.OW * 16u;           // one ring row of one array

    if (warp < FS_NI) {
        // ===================== MMA issuers: tile t -> issuer t % 4 =====================
        const int rank = warp;
        static_assert(FS_NI == 4, "the row advance of FS_NI tiles is found with four comparisons (pooled width >= 128)");
        const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NCOL >> 3) << 17) | ((128u >> 4) << 24);     // M = 128, N = 4 CO
        const uint32_t ahi = 8u | (1u << 14);                  // SBO = 128 B: 8 consecutive slots are one core matrix
        const uint32_t bhi = 16u | (1u << 14);                 // SBO = 256 B between 8-column groups
        const uint32_t b1lo = (bsm >> 4) | (8u << 16), b2lo = ((bsm + (uint32_t)NCOL * 32u) >> 4) | (8u << 16);     // LBO = 128 B between the two K chunks
        const uint32_t albo = (p.arr_bytes >> 4) << 16;        // odd-row array -> even-row array
        int U = U0, gbase = 0, tbase = 0;
        int waited = 0, wphys = 0; uint32_t wphase = 0;        // pair-rows [0, waited) of this CTA's sequence are known to be filled
        FsSeg sg;
        auto wait_rows = [&](int upto) {                       // inclusive, in the CTA's global pair-row numbering
            while (waited <= upto) {
                mbar_wait(bar_full(wphys), wphase);
                ++waited; if (++wphys == p.R) { wphys = 0; wphase ^= 1u; }
            }
        };
        const uint32_t arr16 = arr0 >> 4;
        while (fs_next_seg(p, U, U1, sg)) {
            const int ntiles = sg.ub - sg.ua;
            int k = (rank + FS_NI - tbase % FS_NI) % FS_NI;
            // position of this warp's first tile; afterwards everything advances incrementally (no divisions per tile)
            int pr0 = (int)__umulhi((unsigned)(128 * (sg.ua + k)), p.ow_magic), j0 = 128 * (sg.ua + k) - pr0 * p.OW;
            int ph = (gbase + pr0 - sg.ia) % p.R;              // ring row of pair-row pr0
            int myrel = sg.ia - 1, relph = gbase % p.R;        // pair-rows <= myrel of this frame have been released by this warp; ring row of myrel + 1
            for (; k < ntiles; k += FS_NI) {
                const int t = tbase + k, buf = t % TBUF, use = t / TBUF;
                const int need = min(sg.ib, pr0 + 1 + (j0 + 127 >= p.OW ? 1 : 0));
                const int wnext = j0 + 128 * FS_NI;
                const int adv = (wnext >= p.OW ? 1 : 0) + (wnext >= 2 * p.OW ? 1 : 0) + (wnext >= 3 * p.OW ? 1 : 0) + (wnext >= 4 * p.OW ? 1 : 0);
                // rows no later tile of this warp reads (a row may only be released after it was seen filled: the arrivals on
                // its `empty` barrier must stay behind those of the row that used the ring slot before)
                const int relupto = k + FS_NI < ntiles ? pr0 + adv - 1 : myrel;
                if (rank == 0) FS_STAMP(t / FS_NI, 12);
                FS_WATCH(rank, (t << 8) | 0x10 | (gbase + (max(need, relupto) - sg.ia)) << 16);
                wait_rows(gbase + (max(need, relupto) - sg.ia));
                if (rank == 0) FS_STAMP(t / FS_NI, 13);
                FS_WATCH(rank, (t << 8) | 0x20);
                mbar_wait(bar_tempty(buf), ((uint32_t)use & 1u) ^ 1u);
                if (rank == 0) FS_STAMP(t / FS_NI, 14);
                tc_fence_after();
                if (elect_one()) {
                    const int ph2 = ph + 1 == p.R ? 0 : ph + 1;
                    const uint32_t d = tmem_base + (uint32_t)buf * (uint32_t)NCOL;
                    const uint32_t s1 = arr16 + (uint32_t)(ph * p.OW + j0), s2 = arr16 + (uint32_t)(ph2 * p.OW + j0);
                    umma_i8_lohi<false>(d, s1 | albo, ahi, b1lo, bhi, idesc);           // input rows 2Y - 1, 2Y
                    umma_i8_lohi<true>(d, s2 | albo, ahi, b2lo, bhi, idesc);            // input rows 2Y + 1, 2Y + 2
                    umma_commit(bar_tfull(buf));
                    int rp = relph;
                    for (int r = myrel + 1; r <= relupto; ++r) { umma_commit(bar_empty(rp)); rp = rp + 1 == p.R ? 0 : rp + 1; }
                }
                __syncwarp();
                if (rank == 0) FS_STAMP(t / FS_NI, 15);
                FS_WATCH(rank, (t << 8) | 0x30);
                if (relupto > myrel) { relph += relupto - myrel; if (relph >= p.R) relph -= p.R; myrel = relupto; }
                j0 = wnext - adv * p.OW; pr0 += adv; ph += adv; if (ph >= p.R) ph -= p.R;
            }
            // the rest of the frame segment's rows (after this warp's last tile)
            FS_WATCH(rank, 0x40 | (gbase + (sg.ib - sg.ia)) << 16);
            wait_rows(gbase + (sg.ib - sg.ia));
            if (elect_one()) {
                int rp = relph;
                for (int r = myrel + 1; r <= sg.ib; ++r) { umma_commit(bar_empty(rp)); rp = rp + 1 == p.R ? 0 : rp + 1; }
            }
            __syncwarp();
            gbase += sg.ib - sg.ia + 1;
            tbase += ntiles;
        }
    } else if (warp == FS_LW) {
        // ===================== raw-row loader: one bulk copy per pair-row =====================
        if (lane == 0) {
            int U = U0, rs = 0; uint32_t rphase = 0;
            FsSeg sg;
            const uint8_t *src = reinterpret_cast<const uint8_t *>(p.src);
            while (fs_next_seg(p, U, U1, sg)) {
                for (int r = sg.ia; r <= sg.ib; ++r) {
                    FS_WATCH(4, (r << 16) | rs);
                    mbar_wait_hint(bar_rawempty(rs), rphase ^ 1u);
                    const int ya = 2 * r - 1, yb = 2 * r;
                    const bool va = ya >= 0, vb = yb < p.H;
                    const uint32_t dst = raw0 + (uint32_t)rs * raw_slot_bytes;
                    const uint8_t *row_a = src + ((size_t)sg.img * p.H + (va ? ya : 0)) * p.row_bytes;
                    if (va && vb) {
                        mbar_expect_tx(bar_rawfull(rs), 2u * p.row_bytes);
                        bulk_load_1d(dst, row_a, 2u * p.row_bytes, bar_rawfull(rs));
                    } else if (va) {
                        mbar_expect_tx(bar_rawfull(rs), p.row_bytes);
                        bulk_load_1d(dst, row_a, p.row_bytes, bar_rawfull(rs));
                    } else {
                        mbar_expect_tx(bar_rawfull(rs), p.row_bytes);
                        bulk_load_1d(dst + p.row_bytes, row_a, p.row_bytes, bar_rawfull(rs));      // pair-row 0: row 0 is the even row
                    }
                    if (++rs == FS_RAWR) { rs = 0; rphase ^= 1u; }
                }
            }
        }
    } else if (warp >= FS_BW0 && warp < FS_BW0 + FS_NBW) {
        // ===================== slot builders: warp b fills pair-rows b, b + 8, ... of the CTA's sequence =====================
        const int bw = warp - FS_BW0;
        int U = U0, gl = 0;                                    // gl: index of the current pair-row in the CTA's sequence
        const int team = bw >> 1, rho = bw & 1;                // this warp's rows of the sequence and its input row of a pair-row
        int mine = team, phys = team % p.R, rs = team; uint32_t rphase = 0, phase = (uint32_t)(team / p.R) & 1u;
        static_assert(FS_NTEAM <= FS_RAWR, "a team's first row has a raw slot");
        FsSeg sg;
        const uint32_t mirror_off = (uint32_t)p.R * row_pitch;
        const int lane_j = lane - 1;                           // pass s, lane l <-> pixel pair 30 s + l - 1 (lanes 0 and 31 only feed their neighbours)
        const bool lane_st = lane >= 1 && lane <= FS_SEGW;
        const int jmax = p.OW - 1;
        while (fs_next_seg(p, U, U1, sg)) {
            const int gend = gl + (sg.ib - sg.ia + 1);             // the segment's pair-rows are gl .. gend - 1 of the CTA's sequence
            for (; mine < gend; ) {
                const int r = sg.ia + (mine - gl);
                const int gl_row = mine;
                FS_STAMP_B(0);
                FS_WATCH(5 + bw, (gl_row << 8) | 1);
                mbar_wait_hint(bar_rawfull(rs), rphase);
                FS_WATCH(5 + bw, (gl_row << 8) | 2);
                FS_STAMP_B(1);
                mbar_wait_hint(bar_empty(phys), phase ^ 1u);
                FS_STAMP_B(2);
                FS_WATCH(5 + bw, (gl_row << 8) | 3);
                const uint8_t *rawp = s_rawp + (size_t)rs * raw_slot_bytes;
                const bool mirror = phys < p.MR;
                {
                    const bool rowok = (unsigned)(2 * r - 1 + rho) < (unsigned)p.H;
                    const uint8_t *rr = rawp + rho * p.row_bytes;
                    const uint32_t dst0 = arr0 + (uint32_t)rho * p.arr_bytes + (uint32_t)(phys * p.OW + lane_j) * 16u;
#pragma unroll 1
                    for (int s0 = 0; s0 < p.segs; s0 += 4) {
                        unsigned wl[4], wh[4];
                        // all loads of four passes first, from clamped (always valid) addresses: no branches, the table lookups of
                        // the four passes overlap.  Outside the frame: code 0x1000 -> table entry 4096 = 0 = the zero padding
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int jj = FS_SEGW * (s0 + i) + lane_j;
                            const bool ok = rowok && (unsigned)jj <= (unsigned)jmax;
                            const int jc = min(max(jj, 0), jmax);
                            if (SRC == 1) {
                                const unsigned raw = reinterpret_cast<const unsigned *>(rr)[jc];
                                wl[i] = ok ? (raw & 0x0fff0fffu) : 0x10001000u;
                            } else if (SRC == 2) {
                                // two BGR pixels = six bytes at a 2-byte aligned offset: B0 G0 | R0 B1 | G1 R1
                                const unsigned short *h = reinterpret_cast<const unsigned short *>(rr) + 3 * jc;
                                const unsigned h0 = h[0], h1 = h[1], h2 = h[2];
                                wl[i] = h0 | (h1 << 16);                           // B0 G0 R0 B1
                                wh[i] = ok ? (h2 | 0x10000u) : 0u;                 // G1 R1, bit 16 = inside the frame
                            } else {
                                const uint2 v = reinterpret_cast<const uint2 *>(rr)[jc];
                                wl[i] = ok ? v.x : 0u; wh[i] = ok ? v.y : 0u;
                            }
                        }
                        if (SRC == 1) {
#pragma unroll
                            for (int i = 0; i < 4; ++i) { const unsigned c = wl[i]; wl[i] = s_lut[c & 0xffffu]; wh[i] = s_lut[c >> 16]; }
                        }
                        if (SRC == 2) {
                            const unsigned char *t8 = reinterpret_cast<const unsigned char *>(s_lut);       // [R | G | B][256]
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const unsigned a = wl[i], b = wh[i];
                                const unsigned p0 = (unsigned)t8[(a >> 16) & 255u] | ((unsigned)t8[256 + ((a >> 8) & 255u)] << 8) | ((unsigned)t8[512 + (a & 255u)] << 16);
                                const unsigned p1 = (unsigned)t8[(b >> 8) & 255u] | ((unsigned)t8[256 + (b & 255u)] << 8) | ((unsigned)t8[512 + (a >> 24)] << 16);
                                const bool in = (b >> 16) != 0u;
                                wl[i] = in ? p0 : 0u; wh[i] = in ? p1 : 0u;
                            }
                        }
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const unsigned left = __shfl_up_sync(0xffffffffu, wh[i], 1), right = __shfl_down_sync(0xffffffffu, wl[i], 1);
                            const int jj = FS_SEGW * (s0 + i) + lane_j;
                            const bool st = lane_st && jj <= jmax;
                            const uint32_t dst = dst0 + (uint32_t)(FS_SEGW * 16 * (s0 + i));
                            st_shared_v4_if(st, dst, left, wl[i], wh[i], right);            // pixels 2 jj - 1 .. 2 jj + 2
                            if (mirror) st_shared_v4_if(st, dst + mirror_off, left, wl[i], wh[i], right);      // warp-uniform
                        }
                    }
                }
                FS_STAMP_B(3);
                fence_proxy_async();                           // the slots are read by the tensor core (async proxy)
                FS_STAMP_B(4);
                mbar_arrive(bar_full(phys));
                mbar_arrive(bar_rawempty(rs));
                FS_STAMP_B(5);
                FS_WATCH(5 + bw, (gl_row << 8) | 4);
                rs += FS_NTEAM; if (rs >= FS_RAWR) { rs -= FS_RAWR; rphase ^= 1u; }
                mine += FS_NTEAM;
                phys += FS_NTEAM; while (phys >= p.R) { phys -= p.R; phase ^= 1u; }
            }
            gl = gend;
        }
    } else if (warp >= FS_EW0) {
        // ===================== epilogue warps: tile t -> group t % 4 =====================
        const int grp = (warp - FS_EW0) >> 2, q4 = warp & 3;
        unsigned ovf = 0;
        int U = U0, tbase = 0;
        FsSeg sg;
        const EpiPk kp = epi_pack(p.k);                        // the epilogue constants as packed register pairs
        while (fs_next_seg(p, U, U1, sg)) {
            const int ntiles = sg.ub - sg.ua;
            for (int k = (grp - tbase) & (FS_EG - 1); k < ntiles; k += FS_EG) {
                const int t = tbase + k, buf = t % TBUF, use = t / TBUF;
                FS_WATCH(13 + (warp - FS_EW0), (t << 8) | 1);
                mbar_wait_hint(bar_tfull(buf), (uint32_t)use & 1u);
                FS_WATCH(13 + (warp - FS_EW0), (t << 8) | 2);
                if (grp == 0 && q4 == 0) FS_STAMP(t >> 2, 16);
                tc_fence_after();
                const uint32_t taddr = tmem_base + (uint32_t)buf * (uint32_t)NCOL + ((uint32_t)(q4 * 32) << 16);
                const int q = 128 * (sg.ua + k) + q4 * 32 + lane;
                if (p.q.activ) fs_epilogue_tile<EPI, true, CO>(p, kp, taddr, q, sg.img, s_bias, bar_tempty(buf), ovf);
                else fs_epilogue_tile<EPI, false, CO>(p, kp, taddr, q, sg.img, s_bias, bar_tempty(buf), ovf);
                if (grp == 0 && q4 == 0) FS_STAMP(t >> 2, 17);
                FS_WATCH(13 + (warp - FS_EW0), (t << 8) | 3);
            }
            tbase += ntiles;
        }
        if (p.q.contract == CONTRACT_P) {
            ovf = __reduce_add_sync(0xffffffffu, ovf);
            if (lane == 0 && ovf) atomicAdd(p.ovf, ovf);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
static bool fs_enabled()
{
    static const bool on = [] { const char *e = getenv("YOLO_B200_FS"); return e ? atoi(e) != 0 : true; }();
    return on;
}
static unsigned fs_magic(int d) { return (unsigned)(((1ull << 32) + (unsigned)d - 1) / (unsigned)d); }
constexpr uint32_t FS_SMEM_MAX = 227u * 1024u;

// fills the geometry part of p; false = this kernel does not take the layer
static bool fs_plan(const ConvArgs &a, InKind src_kind, const void *src, FsParams &p)
{
    memset(&p, 0, sizeof p);
    if (!fs_enabled() || src_kind == IN_F32) return false;
    if (src_kind == IN_BGR && (a.W % 16)) return false;                 // rows of 3 W bytes are bulk-copied: multiples of 16 bytes
    if (a.cs_in != 4 || (a.cs_out != 16 && a.cs_out != 32) || a.w_rows < a.cs_out || !a.q.pool) return false;
    if (a.H < 2 || a.W < 256 || (a.W % 8)) return false;       // pooled width >= 128: a tile spans at most two pooled rows
    if (((uintptr_t)src & 15) || ((uintptr_t)a.out & 15)) return false;
    p.n_img = a.n; p.H = a.H; p.W = a.W; p.OH = a.H / 2; p.OW = a.W / 2; p.co = a.cs_out;
    const long long ohw = (long long)p.OH * p.OW;
    if ((ohw + 512) * p.OW >= (1ll << 32) || ohw + 512 >= (1ll << 24)) return false;   // multiply-high divisions stay exact
    p.ohw = (int)ohw;
    p.upi = (int)((ohw + 127) / 128);
    const long long total = (long long)p.upi * a.n;
    if (total * p.upi >= (1ll << 32) || total >= (1ll << 31)) return false;
    p.total_units = (int)total;
    p.ow_magic = fs_magic(p.OW); p.upi_magic = fs_magic(p.upi);
    p.MR = (127 + p.OW - 1) / p.OW;                            // = 1
    p.segs = (p.OW + FS_SEGW - 1) / FS_SEGW;
    p.row_bytes = (uint32_t)a.W * (src_kind == IN_RGB444 ? 2u : src_kind == IN_BGR ? 3u : 4u);
    p.off_lut = 2u * 4u * (uint32_t)a.cs_out * 32u;             // the two weight images
    p.off_raw = p.off_lut + (src_kind == IN_RGB444 ? 4112u * 4u : src_kind == IN_BGR ? 768u : 0u);       // 4097 table words / three byte tables
    p.off_bias = p.off_raw + (uint32_t)FS_RAWR * 2u * p.row_bytes;
    p.off_bar = (p.off_bias + 128u + 15u) & ~15u;
    p.off_arr = (p.off_bar + 8u * (2 * FS_RAWR + 2 * FS_RMAX + 2 * FS_TBUF_MAX + 1) + 127u) & ~127u;
    const uint32_t avail = FS_SMEM_MAX - 128u - p.off_arr;
    const uint32_t row2 = 2u * (uint32_t)p.OW * 16u;           // one ring row of the two arrays
    int rows = (int)(avail / row2) - 1;                        // -1: rounding of arr_bytes
    int R = rows - p.MR;
    if (R > FS_RMAX) R = FS_RMAX;
    if (R < 6) return false;
    p.R = R;
    p.arr_bytes = ((uint32_t)(R + p.MR) * (uint32_t)p.OW * 16u + 127u) & ~127u;
    if (2u * p.arr_bytes + p.off_arr + 128u > FS_SMEM_MAX || (p.arr_bytes >> 4) >= (1u << 14)) return false;
    return true;
}

bool conv3x3_fs_supported(const ConvArgs &a, InKind src_kind, const void *src)
{
    FsParams p;
    return fs_plan(a, src_kind, src, p);
}

template <int EPI, int SRC, int CO>
static cudaError_t launch_fs2(const FsParams &p, cudaStream_t st, int sm_count)
{
    const uint32_t smem_bytes = p.off_arr + 2u * p.arr_bytes + 128u;
    static bool attr_set[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_set[dev & 63]) {
        cudaError_t e = cudaFuncSetAttribute(conv3x3_fs_kernel<EPI, SRC, CO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FS_SMEM_MAX);
        if (e != cudaSuccess) return e;
        attr_set[dev & 63] = true;
    }
    const int grid = p.total_units < sm_count ? p.total_units : sm_count;
#ifdef YB_FS_TIMELINE
    FsParams pd = p;
    {
        static long long *dbg = nullptr;
        if (!dbg) cudaMalloc(&dbg, 64 * 24 * sizeof(long long));
        cudaMemsetAsync(dbg, 0, 64 * 24 * sizeof(long long), st);
        pd.dbg = dbg;
    }
    cudaError_t le = launch_pdl(conv3x3_fs_kernel<EPI, SRC, CO>, dim3(grid), dim3(FS_THREADS), smem_bytes, st, pd);
    if (le != cudaSuccess) return le;
    {
        static long long h[64 * 24];
        cudaStreamSynchronize(st);
        cudaMemcpy(h, pd.dbg, sizeof h, cudaMemcpyDeviceToHost);
        const long long t0 = h[0];
        printf("FS timeline OW=%d R=%d units=%d grid=%d (cycles since builder 0's first stamp): n | builder warp 0, row 4n: start raw_ok slot_ok stored fenced published | builder warp 7, row 4n+3: same | issuer0 tile 4n: top rows_ok tmem_ok issued | epi0 tile 4n: tfull_ok done\n", p.OW, p.R, p.total_units, grid);
        for (int i = 0; i < 40; ++i) {
            printf("  %2d |", i);
            for (int j = 0; j < 18; ++j) printf("%s%7lld", (j == 6 || j == 12 || j == 16) ? " |" : "", h[i * 24 + j] - t0);
            printf("\n");
        }
    }
    return cudaGetLastError();
#elif defined(YB_FS_WATCH)
    FsParams pw = p;
    static unsigned *wh = nullptr, *wd = nullptr;
    if (!wh) { cudaHostAlloc((void **)&wh, 148 * 32 * 4, cudaHostAllocMapped); cudaHostGetDevicePointer((void **)&wd, wh, 0); }
    memset(wh, 0, 148 * 32 * 4);
    pw.watch = wd;
    cudaError_t le = launch_pdl(conv3x3_fs_kernel<EPI, SRC, CO>, dim3(grid), dim3(FS_THREADS), smem_bytes, st, pw);
    if (le != cudaSuccess) return le;
    for (int i = 0; i < 300; ++i) { if (cudaStreamQuery(st) == cudaSuccess) return cudaSuccess; struct timespec ts = {0, 10000000}; nanosleep(&ts, nullptr); }
    printf("FS WATCH: kernel not finished after 3 s.  CO=%d SRC=%d OW=%d R=%d units=%d upi=%d grid=%d\n", CO, SRC, p.OW, p.R, p.total_units, p.upi, grid);
    for (int c = 0; c < grid; ++c) {
        printf("cta %3d [%d,%d) iss", c, (int)(((long long)p.total_units * c) / grid), (int)(((long long)p.total_units * (c + 1)) / grid));
        for (int j = 0; j < 4; ++j) printf(" t%u:%02x:r%u", (wh[c * 32 + j] >> 8) & 0xff, wh[c * 32 + j] & 0xff, wh[c * 32 + j] >> 16);
        printf(" | ld r%u s%u | bld", wh[c * 32 + 4] >> 16, wh[c * 32 + 4] & 0xffff);
        for (int j = 0; j < FS_NBW; ++j) printf(" %u:%u", wh[c * 32 + 5 + j] >> 8, wh[c * 32 + 5 + j] & 0xff);
        printf(" | epi");
        for (int j = 0; j < 16; j += 4) printf(" %u:%u", wh[c * 32 + 13 + j] >> 8, wh[c * 32 + 13 + j] & 0xff);
        printf("\n");
        if (c > 12) break;
    }
    fflush(stdout);
    abort();
#else
    return launch_pdl(conv3x3_fs_kernel<EPI, SRC, CO>, dim3(grid), dim3(FS_THREADS), smem_bytes, st, p);
#endif
}

template <int EPI>
static cudaError_t launch_fs(const FsParams &p, InKind src_kind, cudaStream_t st, int sm_count)
{
    if (p.co == 32) return src_kind == IN_RGB444 ? launch_fs2<EPI, IN_RGB444, 32>(p, st, sm_count) : src_kind == IN_BGR ? launch_fs2<EPI, IN_BGR, 32>(p, st, sm_count) : launch_fs2<EPI, IN_INT8, 32>(p, st, sm_count);
    return src_kind == IN_RGB444 ? launch_fs2<EPI, IN_RGB444, 16>(p, st, sm_count) : src_kind == IN_BGR ? launch_fs2<EPI, IN_BGR, 16>(p, st, sm_count) : launch_fs2<EPI, IN_INT8, 16>(p, st, sm_count);
}

cudaError_t conv3x3_fs(const ConvArgs &a, cudaStream_t st, InKind src_kind, const void *src, const void *lut)
{
    if (a.n == 0) return cudaSuccess;
    FsParams p;
    if (!fs_plan(a, src_kind, src, p)) return cudaErrorInvalidValue;
    if (src_kind != IN_INT8 && !lut) return cudaErrorInvalidValue;
    p.src = src; p.lut = (const int *)lut;
    p.wgt = a.wgt; p.bias_sh = a.bias_sh; p.q = a.q; p.out = a.out; p.ovf = a.ovf;
    p.xsplit = a.out_xsplit ? 1 : 0;
    if (p.xsplit && ((p.OW & 1) || p.co != 16)) return cudaErrorInvalidValue;
    static int sms[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!sms[dev & 63]) cudaDeviceGetAttribute(&sms[dev & 63], cudaDevAttrMultiProcessorCount, dev);
    const int sm_count = sms[dev & 63] > 0 ? sms[dev & 63] : 148;
    switch (epi_mode_for(a, &p.k)) {
    case EPI_F_RNE:      return launch_fs<EPI_F_RNE>(p, src_kind, st, sm_count);
    case EPI_F_RNE_NOHI: return launch_fs<EPI_F_RNE_NOHI>(p, src_kind, st, sm_count);
    case EPI_P:          return launch_fs<EPI_P>(p, src_kind, st, sm_count);
    default:             return launch_fs<EPI_GENERIC>(p, src_kind, st, sm_count);
    }
}

}  // namespace yb
