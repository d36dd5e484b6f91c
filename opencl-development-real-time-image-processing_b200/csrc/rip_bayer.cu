// rip_bayer.cu -- 8-bit Bayer raw frames (RIP_FMT_BAYER_RGGB8, _BGGR8, _GRBG8, _GBRG8) demosaiced to colour, or straight to
// the reference's gray, and the same for 10- to 16-bit samples (RIP_FMT_BAYER_RGGB10 ... _GBRG16) and for packed 10- and
// 12-bit samples (RIP_FMT_BAYER_RGGB10P_MIPI ... _GBRG12P_GENICAM); their sections below.
// launch_yuv (rip_yuv.cu) checks the shape and calls launch_bayer.
//
// The demosaic is OpenCV's default (bilinear) cvtColor(COLOR_Bayer**2RGB), bit for bit.  For an interior pixel with raw
// byte c, h the sum of its left and right neighbours, v the sum of the pixels above and below, n = h + v and d the sum of the
// four diagonals:
//     red site:              R = c, G = (n + 2) >> 2, B = (d + 2) >> 2
//     blue site:             B = c, G = (n + 2) >> 2, R = (d + 2) >> 2
//     green site, red row:   G = c, R = (h + 1) >> 1, B = (v + 1) >> 1
//     green site, blue row:  G = c, B = (h + 1) >> 1, R = (v + 1) >> 1
// Border pixels copy their interior neighbour, colour phase included: out(y, x) = out(clamp(y, 1, H-2), clamp(x, 1, W-2)).
// Every output is an average of bytes, so nothing saturates.  Gray and the output stores are rip_decode.cuh's, as for YUV.
//
// x8 kernel (W % 8 == 0, input 8-byte aligned, output 8-byte or, for 4 bytes per pixel, 16-byte aligned): one thread owns an
// even/odd row pair x 8 columns at an even x, so every site's colour role is a compile-time constant.  It loads the raw rows
// above, in and below the pair as one 64-bit word each; the byte left and the byte right of each word come from the
// neighbouring lanes by shuffle (a 32-bit load at the warp's two edge lanes).  A border row pair computes its one source row
// and stores it to both of its rows; the first and last column groups copy pixel 1 to pixel 0 and pixel 6 to pixel 7.
// Any other width (odd W makes a row's colour phase independent of its address) and unaligned buffers or frame strides (an
// odd W * H misaligns every second frame) take the byte-granular kernel: one pixel per thread.  Frames ride in gridDim.y.
#include "rip_decode.cuh"

namespace rip {
namespace {

// the red site's (row, column) in the pattern's top-left 2x2; blue sits diagonally opposite, green on the other two
template <int FMT> struct Pattern;
template <> struct Pattern<RIP_FMT_BAYER_RGGB8> { static constexpr int ry = 0, rx = 0; };
template <> struct Pattern<RIP_FMT_BAYER_BGGR8> { static constexpr int ry = 1, rx = 1; };
template <> struct Pattern<RIP_FMT_BAYER_GRBG8> { static constexpr int ry = 0, rx = 1; };
template <> struct Pattern<RIP_FMT_BAYER_GBRG8> { static constexpr int ry = 1, rx = 0; };

// the colour of one site: red_row / red_col say whether its row / column holds red sites
__device__ __forceinline__ Rgb site(bool red_row, bool red_col, int c, int h, int v, int d)
{
    if (red_row && red_col) return {c, (h + v + 2) >> 2, (d + 2) >> 2};
    if (!red_row && !red_col) return {(d + 2) >> 2, (h + v + 2) >> 2, c};
    if (red_row) return {(h + 1) >> 1, c, (v + 1) >> 1};
    return {(v + 1) >> 1, c, (h + 1) >> 1};
}

// One raw row as seen by a thread: its 8 bytes, and the byte on either side (bits 0..7 of l and r).
struct Row10 {
    uint2 w;
    uint32_t l, r;
};

// byte j of the row, j = -1 .. 8
__device__ __forceinline__ int at(const Row10 &q, int j)
{
    if (j < 0) return (int)q.l;
    if (j > 7) return (int)q.r;
    return (int)(((j < 4 ? q.w.x : q.w.y) >> (8 * (j & 3))) & 0xffu);
}

// Eight output pixels of a source row of colour phase P (0: the pattern's first row), from the raw rows above (a), at (m) and
// below (b) it.  The vertical sums of each column serve v at its own site and d at both neighbours.
template <int OUT, int FMT, int P>
__device__ __forceinline__ void row_x8(uint32_t px[8], const Row10 &a, const Row10 &m, const Row10 &b)
{
    using Pat = Pattern<FMT>;
    int vs[10];
#pragma unroll
    for (int j = 0; j < 10; j++) vs[j] = at(a, j - 1) + at(b, j - 1);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int h = at(m, i - 1) + at(m, i + 1);
        px[i] = pixel_word<OUT>(site(P == Pat::ry, (i & 1) == Pat::rx, at(m, i), h, vs[i + 1], vs[i] + vs[i + 2]));
    }
}

template <int OUT, int FMT>
__global__ void __launch_bounds__(256)
bayer_kernel_x8(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int W, int H, int f0)
{
    constexpr int BPP = OutFmt<OUT>::bpp;
    const int cols = W >> 3, pairs = (H + 1) >> 1;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = u % cols;                       // 8-column group
    const bool live = u / cols < pairs;
    const int y0 = 2 * min(u / cols, pairs - 1);  // spare lanes load a real row pair for the shuffles and store nothing
    const int s0 = min(max(y0, 1), H - 2);        // source row of output row y0
    const int s1 = min(max(y0 + 1, 1), H - 2);    // and of y0 + 1: s0 + 1 inside the frame, s0 in a border pair
    const size_t frame = ((size_t)f0 + blockIdx.y) * W * H;
    const uint8_t *base = in + frame + 8 * c;
    const int lane = threadIdx.x & 31;
    uint2 w[4];   // raw rows s0 - 1 .. s0 + 2 (the last is read only when s1 = s0 + 1)
#pragma unroll
    for (int i = 0; i < 4; i++) w[i] = __ldg(reinterpret_cast<const uint2 *>(base + (size_t)min(s0 - 1 + i, H - 1) * W));
    // the four rows' last bytes and first bytes, one word each: lane - 1 (group c - 1 of the same rows) sends its last bytes
    // as this lane's left halo, lane + 1 its first bytes as the right halo
    uint32_t left = __shfl_up_sync(0xffffffffu, __byte_perm(__byte_perm(w[0].y, w[1].y, 0x0073), __byte_perm(w[2].y, w[3].y, 0x0073), 0x5410), 1);
    uint32_t right = __shfl_down_sync(0xffffffffu, __byte_perm(__byte_perm(w[0].x, w[1].x, 0x0040), __byte_perm(w[2].x, w[3].x, 0x0040), 0x5410), 1);
    if (lane == 0 && c > 0) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const uint32_t b = __ldg(reinterpret_cast<const uint32_t *>(base + (size_t)min(s0 - 1 + i, H - 1) * W - 4)) >> 24;
            left = (left & ~(0xffu << (8 * i))) | b << (8 * i);
        }
    }
    if (lane == 31 && c < cols - 1) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const uint32_t b = __ldg(reinterpret_cast<const uint32_t *>(base + (size_t)min(s0 - 1 + i, H - 1) * W + 8)) & 0xffu;
            right = (right & ~(0xffu << (8 * i))) | b << (8 * i);
        }
    }
    Row10 q[4];
#pragma unroll
    for (int i = 0; i < 4; i++) q[i] = {w[i], (left >> (8 * i)) & 0xffu, (right >> (8 * i)) & 0xffu};
    uint8_t *o = out + (frame + (size_t)y0 * W + 8 * c) * BPP;
    const size_t next_row = (size_t)W * BPP;
    uint32_t px[8];
    if (s0 & 1) row_x8<OUT, FMT, 1>(px, q[0], q[1], q[2]);
    else row_x8<OUT, FMT, 0>(px, q[0], q[1], q[2]);
    if (c == 0) px[0] = px[1];
    if (c == cols - 1) px[7] = px[6];
    if (live) {
        store_x8<OUT>(o, px);
        if (s1 == s0 && y0 + 1 < H) store_x8<OUT>(o + next_row, px);
    }
    if (s1 != s0) {   // row y0 + 1 inside the frame: s0 is even, s1 odd
        row_x8<OUT, FMT, 1>(px, q[1], q[2], q[3]);
        if (c == 0) px[0] = px[1];
        if (c == cols - 1) px[7] = px[6];
        if (live) store_x8<OUT>(o + next_row, px);
    }
}

// any W, H >= 3, any alignment: one pixel per thread, byte loads and stores
template <int OUT, int FMT>
__global__ void __launch_bounds__(256)
bayer_kernel_x1(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int W, int H, int f0)
{
    using Pat = Pattern<FMT>;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = u / W, x = u - y * W;
    if (y >= H) return;
    const size_t frame = ((size_t)f0 + blockIdx.y) * W * H;
    const int ys = min(max(y, 1), H - 2), xs = min(max(x, 1), W - 2);
    const uint8_t *p = in + frame + (size_t)ys * W + xs;
    const int h = __ldg(p - 1) + __ldg(p + 1), v = __ldg(p - W) + __ldg(p + W);
    const int d = __ldg(p - W - 1) + __ldg(p - W + 1) + __ldg(p + W - 1) + __ldg(p + W + 1);
    const Rgb rgb = site((ys & 1) == Pat::ry, (xs & 1) == Pat::rx, __ldg(p), h, v, d);
    store_px<OUT>(out + (frame + (size_t)y * W + x) * OutFmt<OUT>::bpp, pixel_word<OUT>(rgb));
}

// ---- 10- to 16-bit samples (RIP_FMT_BAYER_RGGB10 ... _GBRG16): W*H little-endian 16-bit words per frame, LSB-aligned ------
// The decode is OpenCV's cvtColor(COLOR_Bayer**2RGB) on the CV_16U frame followed by convertTo(CV_8U, 1.0 / 2^shift), with
// shift = bits - 8: the same formulas on the full 16-bit samples, then each channel divided by 2^shift, rounded half to even
// and saturated (a full-scale 10-bit 1023 gives 255.75, so 256, so 255; padding bits above the depth are used as they are).
// The sums stay in 32-bit lanes (four 16-bit samples need 18 bits).  The pattern and the output are template parameters, as
// above; the shift is a kernel argument, so the four depths share one kernel per pattern and output.

// v / 2^shift rounded half to even, for shift >= 1 (the saturation is pack4's); half_m1 = 2^(shift - 1) - 1
__device__ __forceinline__ int reduce16(int v, int shift, int half_m1) { return (v + half_m1 + ((v >> shift) & 1)) >> shift; }

__device__ __forceinline__ Rgb reduce16(const Rgb &p, int shift, int half_m1)
{
    return {reduce16(p.r, shift, half_m1), reduce16(p.g, shift, half_m1), reduce16(p.b, shift, half_m1)};
}

// One raw row as seen by a thread: its 8 samples (two per word, low half first), and the sample on either side.
struct Row16 {
    uint4 w;
    uint32_t l, r;
};

// sample j of the row, j = -1 .. 8
__device__ __forceinline__ int at(const Row16 &q, int j)
{
    if (j < 0) return (int)q.l;
    if (j > 7) return (int)q.r;
    const uint32_t word = j < 2 ? q.w.x : j < 4 ? q.w.y : j < 6 ? q.w.z : q.w.w;
    return (int)((word >> (16 * (j & 1))) & 0xffffu);
}

// row_x8 for 16-bit samples: the same sums and sites, then the reduction to 8 bits.  Row is any type with an at(row, j) for
// j = -1 .. 8: Row16 here, the packed rows of the next section.
template <int OUT, int FMT, int P, class Row>
__device__ __forceinline__ void row16_x8(uint32_t px[8], const Row &a, const Row &m, const Row &b, int shift, int half_m1)
{
    using Pat = Pattern<FMT>;
    int vs[10];
#pragma unroll
    for (int j = 0; j < 10; j++) vs[j] = at(a, j - 1) + at(b, j - 1);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int h = at(m, i - 1) + at(m, i + 1);
        const Rgb rgb = site(P == Pat::ry, (i & 1) == Pat::rx, at(m, i), h, vs[i + 1], vs[i] + vs[i + 2]);
        px[i] = pixel_word<OUT>(reduce16(rgb, shift, half_m1));
    }
}

// bayer_kernel_x8's shape for 16-bit samples (W % 8 == 0, input 16-byte aligned, output as there): a row pair x 8 columns per
// thread, one 128-bit load per raw row, and the halo samples of the four rows in two shuffles each way (rows 0, 1 and rows
// 2, 3 share a word), the warp's two edge lanes loading theirs.  FMT is the 8-bit code of the same pattern.
template <int OUT, int FMT>
__global__ void __launch_bounds__(256)
bayer16_kernel_x8(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int W, int H, int f0, int shift)
{
    constexpr int BPP = OutFmt<OUT>::bpp;
    const int cols = W >> 3, pairs = (H + 1) >> 1;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = u % cols;
    const bool live = u / cols < pairs;
    const int y0 = 2 * min(u / cols, pairs - 1);
    const int s0 = min(max(y0, 1), H - 2);
    const int s1 = min(max(y0 + 1, 1), H - 2);
    const size_t frame = ((size_t)f0 + blockIdx.y) * W * H;   // in pixels
    const uint16_t *base = reinterpret_cast<const uint16_t *>(in) + frame + 8 * c;
    const int lane = threadIdx.x & 31;
    uint4 w[4];   // raw rows s0 - 1 .. s0 + 2
#pragma unroll
    for (int i = 0; i < 4; i++) w[i] = __ldg(reinterpret_cast<const uint4 *>(base + (size_t)min(s0 - 1 + i, H - 1) * W));
    // halo words: the last samples (left halo of lane + 1) or first samples (right halo of lane - 1) of rows 0, 1 and of 2, 3
    uint32_t left01 = __shfl_up_sync(0xffffffffu, __byte_perm(w[0].w, w[1].w, 0x7632), 1);
    uint32_t left23 = __shfl_up_sync(0xffffffffu, __byte_perm(w[2].w, w[3].w, 0x7632), 1);
    uint32_t right01 = __shfl_down_sync(0xffffffffu, __byte_perm(w[0].x, w[1].x, 0x5410), 1);
    uint32_t right23 = __shfl_down_sync(0xffffffffu, __byte_perm(w[2].x, w[3].x, 0x5410), 1);
    if (lane == 0 && c > 0) {   // samples -2, -1 of each row; keep -1
        uint32_t e[4];
#pragma unroll
        for (int i = 0; i < 4; i++) e[i] = __ldg(reinterpret_cast<const uint32_t *>(base + (size_t)min(s0 - 1 + i, H - 1) * W - 2));
        left01 = __byte_perm(e[0], e[1], 0x7632);
        left23 = __byte_perm(e[2], e[3], 0x7632);
    }
    if (lane == 31 && c < cols - 1) {   // samples 8, 9 of each row; keep 8
        uint32_t e[4];
#pragma unroll
        for (int i = 0; i < 4; i++) e[i] = __ldg(reinterpret_cast<const uint32_t *>(base + (size_t)min(s0 - 1 + i, H - 1) * W + 8));
        right01 = __byte_perm(e[0], e[1], 0x5410);
        right23 = __byte_perm(e[2], e[3], 0x5410);
    }
    const Row16 q[4] = {{w[0], left01 & 0xffffu, right01 & 0xffffu}, {w[1], left01 >> 16, right01 >> 16},
                        {w[2], left23 & 0xffffu, right23 & 0xffffu}, {w[3], left23 >> 16, right23 >> 16}};
    const int half_m1 = (1 << (shift - 1)) - 1;
    uint8_t *o = out + (frame + (size_t)y0 * W + 8 * c) * BPP;
    const size_t next_row = (size_t)W * BPP;
    uint32_t px[8];
    if (s0 & 1) row16_x8<OUT, FMT, 1>(px, q[0], q[1], q[2], shift, half_m1);
    else row16_x8<OUT, FMT, 0>(px, q[0], q[1], q[2], shift, half_m1);
    if (c == 0) px[0] = px[1];
    if (c == cols - 1) px[7] = px[6];
    if (live) {
        store_x8<OUT>(o, px);
        if (s1 == s0 && y0 + 1 < H) store_x8<OUT>(o + next_row, px);
    }
    if (s1 != s0) {
        row16_x8<OUT, FMT, 1>(px, q[1], q[2], q[3], shift, half_m1);
        if (c == 0) px[0] = px[1];
        if (c == cols - 1) px[7] = px[6];
        if (live) store_x8<OUT>(o + next_row, px);
    }
}

// any W, H >= 3, any alignment (odd byte addresses included): one pixel per thread, each sample from two byte loads
template <int OUT, int FMT>
__global__ void __launch_bounds__(256)
bayer16_kernel_x1(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int W, int H, int f0, int shift)
{
    using Pat = Pattern<FMT>;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = u / W, x = u - y * W;
    if (y >= H) return;
    const size_t frame = ((size_t)f0 + blockIdx.y) * W * H;
    const int ys = min(max(y, 1), H - 2), xs = min(max(x, 1), W - 2);
    const uint8_t *p = in + 2 * (frame + (size_t)ys * W + xs);
    const auto at = [p](ptrdiff_t i) { return (int)__ldg(p + 2 * i) | (int)__ldg(p + 2 * i + 1) << 8; };
    const int h = at(-1) + at(1), v = at(-W) + at(W);
    const int d = at(-W - 1) + at(-W + 1) + at(W - 1) + at(W + 1);
    const Rgb rgb = site((ys & 1) == Pat::ry, (xs & 1) == Pat::rx, at(0), h, v, d);
    store_px<OUT>(out + (frame + (size_t)y * W + x) * OutFmt<OUT>::bpp, pixel_word<OUT>(reduce16(rgb, shift, (1 << (shift - 1)) - 1)));
}

// ---- packed 10- and 12-bit samples (RIP_FMT_BAYER_RGGB10P_MIPI ... _GBRG12P_GENICAM): W*b/8 bytes per row, no padding -------
// MIPI CSI-2 RAW10: 4 pixels in 5 bytes; bytes 0-3 hold bits 9..2 of pixels 0-3, byte 4 bits 1..0 of pixel i at 2i+1..2i.
// MIPI CSI-2 RAW12: 2 pixels in 3 bytes; bytes 0-1 hold bits 11..4 of pixels 0-1, byte 2 bits 3..0 of pixel 0 (low nibble)
// and of pixel 1 (high nibble).  GenICam BayerRG10p / 12p ...: an LSB-first bit stream, pixel i at stream bits b*i .. b*i+b-1,
// stream bit k at bit k % 8 of byte k / 8.  The samples are unpacked in registers and go through the 16-bit path above
// (row16_x8, site, reduce16 with shift b - 8), so the decode is that of RIP_FMT_BAYER_<pattern>10 / 12 on the unpacked frame.

// bits pos .. pos + n - 1 (n <= 25) of the little-endian word array w; pos is a compile-time constant after unrolling
template <int NW>
__device__ __forceinline__ int bits_at(const uint32_t (&w)[NW], int pos, int n)
{
    const int j = pos >> 5, s = pos & 31;
    const uint32_t v = s + n <= 32 ? w[j] >> s : __funnelshift_r(w[j], w[min(j + 1, NW - 1)], s);
    return (int)(v & ((1u << n) - 1));
}

// sample k (0 .. 15) of 16 columns packed at BITS bits in BITS / 2 words
template <int BITS, bool GENICAM>
__device__ __forceinline__ int unpack_at(const uint32_t (&w)[BITS / 2], int k)
{
    if constexpr (GENICAM) return bits_at(w, BITS * k, BITS);
    constexpr int per = BITS == 10 ? 4 : 2;   // MIPI: per pixels in per + 1 bytes, the low bits in the last
    const int g = 8 * (per + 1) * (k / per), i = k % per;
    return bits_at(w, g + 8 * i, 8) << (BITS - 8) | bits_at(w, g + 8 * per + (BITS - 8) * i, BITS - 8);
}

// One packed raw row as seen by a thread: its 16 columns and the sample on either side
template <int BITS, bool GENICAM>
struct PackedRow {
    uint32_t w[BITS / 2];
    int l, r;
};

// the half (columns 8*HALF .. 8*HALF + 7) of a packed row that one row16_x8 call reads
template <int BITS, bool GENICAM, int HALF>
struct PackedHalf {
    const PackedRow<BITS, GENICAM> &q;
};

// sample j of the half, j = -1 .. 8
template <int BITS, bool GENICAM, int HALF>
__device__ __forceinline__ int at(const PackedHalf<BITS, GENICAM, HALF> &h, int j)
{
    const int k = 8 * HALF + j;
    if (k < 0) return h.q.l;
    if (k > 15) return h.q.r;
    return unpack_at<BITS, GENICAM>(h.q.w, k);
}

// Columns 8*HALF .. 8*HALF + 7 of the thread's row pair, stored before the other half is computed (so that only one half's
// pixels are live); the first and last column groups of a row copy pixel 1 to pixel 0 and pixel 14 to pixel 15.
template <int OUT, int FMT, int HALF, int BITS, bool GENICAM>
__device__ __forceinline__ void packed_half_x8(uint8_t *o, size_t next_row, const PackedRow<BITS, GENICAM> (&q)[4], int s0, int s1,
                                               bool store0, bool store1, bool edge)
{
    using Half = PackedHalf<BITS, GENICAM, HALF>;
    constexpr int shift = BITS - 8, half_m1 = (1 << (BITS - 9)) - 1, from = HALF ? 6 : 1, to = HALF ? 7 : 0;
    o += 8 * HALF * OutFmt<OUT>::bpp;
    uint32_t px[8];
    if (s0 & 1) row16_x8<OUT, FMT, 1>(px, Half{q[0]}, Half{q[1]}, Half{q[2]}, shift, half_m1);
    else row16_x8<OUT, FMT, 0>(px, Half{q[0]}, Half{q[1]}, Half{q[2]}, shift, half_m1);
    if (edge) px[to] = px[from];
    if (store0) store_x8<OUT>(o, px);
    if (store1 && s1 == s0) store_x8<OUT>(o + next_row, px);   // a border pair: both rows copy the one source row
    if (s1 != s0) {
        row16_x8<OUT, FMT, 1>(px, Half{q[1]}, Half{q[2]}, Half{q[3]}, shift, half_m1);
        if (edge) px[to] = px[from];
        if (store1) store_x8<OUT>(o + next_row, px);
    }
}

// bayer16_kernel_x8's shape for packed samples (W % 16 == 0, input 4-byte aligned, output as there): a row
// pair x 16 columns per thread, whose packed bytes (2*BITS: 20 or 24) are whole words; BITS / 2 32-bit loads per raw row.  The
// halo samples of the four rows travel in two shuffles each way (rows 0, 1 and rows 2, 3 share a word); the warp's two edge
// lanes load the neighbouring group's last word (sample 15 lies in it) or first two words (sample 0).
template <int OUT, int FMT, int BITS, bool GENICAM>
__global__ void __launch_bounds__(256)
bayer_packed_kernel_x16(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int W, int H, int f0)
{
    constexpr int BPP = OutFmt<OUT>::bpp, NW = BITS / 2;
    const int cols = W >> 4, pairs = (H + 1) >> 1;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = u % cols;
    const bool live = u / cols < pairs;
    const int y0 = 2 * min(u / cols, pairs - 1);
    const int s0 = min(max(y0, 1), H - 2);
    const int s1 = min(max(y0 + 1, 1), H - 2);
    const size_t frame = (size_t)f0 + blockIdx.y, row_bytes = (size_t)W * BITS / 8;
    const uint8_t *base = in + frame * H * row_bytes + (size_t)c * 4 * NW;
    const int lane = threadIdx.x & 31;
    PackedRow<BITS, GENICAM> q[4];   // raw rows s0 - 1 .. s0 + 2
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint32_t *p = reinterpret_cast<const uint32_t *>(base + (size_t)min(s0 - 1 + i, H - 1) * row_bytes);
#pragma unroll
        for (int k = 0; k < NW; k++) q[i].w[k] = __ldg(p + k);
    }
    uint32_t left01 = __shfl_up_sync(0xffffffffu, unpack_at<BITS, GENICAM>(q[0].w, 15) | unpack_at<BITS, GENICAM>(q[1].w, 15) << 16, 1);
    uint32_t left23 = __shfl_up_sync(0xffffffffu, unpack_at<BITS, GENICAM>(q[2].w, 15) | unpack_at<BITS, GENICAM>(q[3].w, 15) << 16, 1);
    uint32_t right01 = __shfl_down_sync(0xffffffffu, unpack_at<BITS, GENICAM>(q[0].w, 0) | unpack_at<BITS, GENICAM>(q[1].w, 0) << 16, 1);
    uint32_t right23 = __shfl_down_sync(0xffffffffu, unpack_at<BITS, GENICAM>(q[2].w, 0) | unpack_at<BITS, GENICAM>(q[3].w, 0) << 16, 1);
    int e[4];
    if (lane == 0 && c > 0) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const uint32_t *p = reinterpret_cast<const uint32_t *>(base + (size_t)min(s0 - 1 + i, H - 1) * row_bytes);
            uint32_t g[NW] = {};
            g[NW - 1] = __ldg(p - 1);
            e[i] = unpack_at<BITS, GENICAM>(g, 15);
        }
        left01 = e[0] | e[1] << 16;
        left23 = e[2] | e[3] << 16;
    }
    if (lane == 31 && c < cols - 1) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const uint32_t *p = reinterpret_cast<const uint32_t *>(base + (size_t)min(s0 - 1 + i, H - 1) * row_bytes);
            uint32_t g[NW] = {};
            g[0] = __ldg(p + NW);
            g[1] = __ldg(p + NW + 1);
            e[i] = unpack_at<BITS, GENICAM>(g, 0);
        }
        right01 = e[0] | e[1] << 16;
        right23 = e[2] | e[3] << 16;
    }
    q[0].l = left01 & 0xffffu, q[1].l = left01 >> 16, q[2].l = left23 & 0xffffu, q[3].l = left23 >> 16;
    q[0].r = right01 & 0xffffu, q[1].r = right01 >> 16, q[2].r = right23 & 0xffffu, q[3].r = right23 >> 16;
    uint8_t *o = out + ((frame * H + y0) * W + 16 * c) * BPP;
    const size_t next_row = (size_t)W * BPP;
    const bool store1 = live && y0 + 1 < H;
    packed_half_x8<OUT, FMT, 0>(o, next_row, q, s0, s1, live, store1, c == 0);
    packed_half_x8<OUT, FMT, 1>(o, next_row, q, s0, s1, live, store1, c == cols - 1);
}

// any legal W, H >= 3, any alignment: one pixel per thread, each sample from the one or two bytes that hold it
template <int OUT, int FMT>
__global__ void __launch_bounds__(256)
bayer_packed_kernel_x1(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int W, int H, int f0, int bits, bool genicam)
{
    using Pat = Pattern<FMT>;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = u / W, x = u - y * W;
    if (y >= H) return;
    const size_t frame = (size_t)f0 + blockIdx.y;
    const ptrdiff_t row_bytes = (ptrdiff_t)W * bits / 8;
    const int ys = min(max(y, 1), H - 2), xs = min(max(x, 1), W - 2);
    const uint8_t *p = in + (ptrdiff_t)(frame * H + ys) * row_bytes;
    const int lo_bits = bits - 8, lo_mask = (1 << lo_bits) - 1;
    const auto at = [=](int dy, int sx) {
        const uint8_t *r = p + dy * row_bytes;
        if (genicam) {
            const size_t bit = (size_t)sx * bits;
            const int v = (int)__ldg(r + (bit >> 3)) | (int)__ldg(r + (bit >> 3) + 1) << 8;
            return (v >> (bit & 7)) & ((1 << bits) - 1);
        }
        const int per = bits == 10 ? 4 : 2, g = sx / per, i = sx - g * per;   // MIPI: per pixels in per + 1 bytes
        const uint8_t *grp = r + (size_t)g * (per + 1);
        return (int)__ldg(grp + i) << lo_bits | ((int)__ldg(grp + per) >> (lo_bits * i) & lo_mask);
    };
    const int h = at(0, xs - 1) + at(0, xs + 1), v = at(-1, xs) + at(1, xs);
    const int d = at(-1, xs - 1) + at(-1, xs + 1) + at(1, xs - 1) + at(1, xs + 1);
    const Rgb rgb = site((ys & 1) == Pat::ry, (xs & 1) == Pat::rx, at(0, xs), h, v, d);
    store_px<OUT>(out + ((frame * H + y) * W + x) * OutFmt<OUT>::bpp, pixel_word<OUT>(reduce16(rgb, lo_bits, (1 << (lo_bits - 1)) - 1)));
}

template <int OUT, int FMT>
int launch_packed(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames, int bits, bool genicam)
{
    const uintptr_t out_align = OutFmt<OUT>::bpp == 4 ? 15u : 7u;
    // The word loads need W % 16 == 0 and a 4-byte aligned input.  Unlike the 8- and 16-bit kernels, no frame stride can then
    // misalign them: a row of 16-column groups is 20 or 24 bytes per group, so every row and frame starts on a word.
    const bool x16 = (W & 15) == 0 && (reinterpret_cast<uintptr_t>(in) & 3u) == 0 && (reinterpret_cast<uintptr_t>(out) & out_align) == 0;
    const long long units = x16 ? (long long)((H + 1) / 2) * (W / 16) : (long long)H * W;   // threads per frame
    const dim3 block(256);
    for (int f0 = 0; f0 < n_frames; f0 += 65535) {
        const dim3 grid((unsigned)((units + 255) / 256), (unsigned)min(n_frames - f0, 65535));
        if (!x16) bayer_packed_kernel_x1<OUT, FMT><<<grid, block, 0, s>>>(in, out, W, H, f0, bits, genicam);
        else if (bits == 10 && genicam) bayer_packed_kernel_x16<OUT, FMT, 10, true><<<grid, block, 0, s>>>(in, out, W, H, f0);
        else if (bits == 10) bayer_packed_kernel_x16<OUT, FMT, 10, false><<<grid, block, 0, s>>>(in, out, W, H, f0);
        else if (genicam) bayer_packed_kernel_x16<OUT, FMT, 12, true><<<grid, block, 0, s>>>(in, out, W, H, f0);
        else bayer_packed_kernel_x16<OUT, FMT, 12, false><<<grid, block, 0, s>>>(in, out, W, H, f0);
        RIP_LAUNCH_CHECK();
    }
    return RIP_OK;
}

// shift: bits per sample - 8; 0 = 8-bit samples.  packing: BAYER_UNPACKED, or the layout of packed samples
template <int OUT, int FMT>
int launch_t(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames, int shift, int packing)
{
    if (packing != BAYER_UNPACKED) return launch_packed<OUT, FMT>(s, in, out, W, H, n_frames, shift + 8, packing == BAYER_GENICAM);
    const uintptr_t in_align = shift ? 15u : 7u, out_align = OutFmt<OUT>::bpp == 4 ? 15u : 7u;
    const bool x8 = (W & 7) == 0 && (reinterpret_cast<uintptr_t>(in) & in_align) == 0 && (reinterpret_cast<uintptr_t>(out) & out_align) == 0;
    const long long units = x8 ? (long long)((H + 1) / 2) * (W / 8) : (long long)H * W;   // threads per frame
    const dim3 block(256);
    for (int f0 = 0; f0 < n_frames; f0 += 65535) {
        const dim3 grid((unsigned)((units + 255) / 256), (unsigned)min(n_frames - f0, 65535));
        if (shift == 0) {
            if (x8) bayer_kernel_x8<OUT, FMT><<<grid, block, 0, s>>>(in, out, W, H, f0);
            else bayer_kernel_x1<OUT, FMT><<<grid, block, 0, s>>>(in, out, W, H, f0);
        } else {
            if (x8) bayer16_kernel_x8<OUT, FMT><<<grid, block, 0, s>>>(in, out, W, H, f0, shift);
            else bayer16_kernel_x1<OUT, FMT><<<grid, block, 0, s>>>(in, out, W, H, f0, shift);
        }
        RIP_LAUNCH_CHECK();
    }
    return RIP_OK;
}

template <int FMT>
int launch_fmt(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames, YuvOut to, int shift, int packing)
{
    switch (to) {
    case YUV_TO_RGB: return launch_t<YUV_TO_RGB, FMT>(s, in, out, W, H, n_frames, shift, packing);
    case YUV_TO_BGR: return launch_t<YUV_TO_BGR, FMT>(s, in, out, W, H, n_frames, shift, packing);
    case YUV_TO_RGBA: return launch_t<YUV_TO_RGBA, FMT>(s, in, out, W, H, n_frames, shift, packing);
    case YUV_TO_BGRA: return launch_t<YUV_TO_BGRA, FMT>(s, in, out, W, H, n_frames, shift, packing);
    case YUV_TO_GRAY: return launch_t<YUV_TO_GRAY, FMT>(s, in, out, W, H, n_frames, shift, packing);
    case YUV_TO_GRAY_RGBA: return launch_t<YUV_TO_GRAY_RGBA, FMT>(s, in, out, W, H, n_frames, shift, packing);
    }
    return fail(RIP_EINVAL, "Bayer decode: bad output %d", (int)to);
}

}  // namespace

// Every Bayer code is routed by its row to the kernels of its pattern (the 8-bit code), its depth (the shift) and its
// packing; anything else is an error, never a default pattern.
int launch_bayer(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames, int in_format, YuvOut to)
{
    const Format *f = format_of(in_format);
    switch (f ? f->pattern : -1) {
    case 0: return launch_fmt<RIP_FMT_BAYER_RGGB8>(s, in, out, W, H, n_frames, to, f->bits - 8, f->packing);
    case 1: return launch_fmt<RIP_FMT_BAYER_BGGR8>(s, in, out, W, H, n_frames, to, f->bits - 8, f->packing);
    case 2: return launch_fmt<RIP_FMT_BAYER_GRBG8>(s, in, out, W, H, n_frames, to, f->bits - 8, f->packing);
    case 3: return launch_fmt<RIP_FMT_BAYER_GBRG8>(s, in, out, W, H, n_frames, to, f->bits - 8, f->packing);
    }
    return fail(RIP_EINVAL, "Bayer decode: input format %d is not a Bayer format", in_format);
}

}  // namespace rip
