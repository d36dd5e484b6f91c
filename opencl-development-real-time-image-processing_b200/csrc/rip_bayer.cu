// rip_bayer.cu -- 8-bit Bayer raw frames (RIP_FMT_BAYER_RGGB8, _BGGR8, _GRBG8, _GBRG8) demosaiced to colour, or straight to
// the reference's gray, and the same for 10- to 16-bit samples (RIP_FMT_BAYER_RGGB10 ... _GBRG16; their section below).
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

// row_x8 for 16-bit samples: the same sums and sites, then the reduction to 8 bits
template <int OUT, int FMT, int P>
__device__ __forceinline__ void row16_x8(uint32_t px[8], const Row16 &a, const Row16 &m, const Row16 &b, int shift, int half_m1)
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

// shift: bits per sample - 8; 0 = 8-bit samples
template <int OUT, int FMT>
int launch_t(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames, int shift)
{
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
int launch_fmt(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames, YuvOut to, int shift)
{
    switch (to) {
    case YUV_TO_RGB: return launch_t<YUV_TO_RGB, FMT>(s, in, out, W, H, n_frames, shift);
    case YUV_TO_BGR: return launch_t<YUV_TO_BGR, FMT>(s, in, out, W, H, n_frames, shift);
    case YUV_TO_RGBA: return launch_t<YUV_TO_RGBA, FMT>(s, in, out, W, H, n_frames, shift);
    case YUV_TO_BGRA: return launch_t<YUV_TO_BGRA, FMT>(s, in, out, W, H, n_frames, shift);
    case YUV_TO_GRAY: return launch_t<YUV_TO_GRAY, FMT>(s, in, out, W, H, n_frames, shift);
    case YUV_TO_GRAY_RGBA: return launch_t<YUV_TO_GRAY_RGBA, FMT>(s, in, out, W, H, n_frames, shift);
    }
    return fail(RIP_EINVAL, "Bayer decode: bad output %d", (int)to);
}

}  // namespace

// Every Bayer code is routed by name to the kernels of its pattern (the 8-bit code) and its depth (the shift); anything
// else is an error, never a default pattern.
int launch_bayer(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames, int in_format, YuvOut to)
{
    const int shift = bayer_bits(in_format) - 8;
    switch (in_format) {
    case RIP_FMT_BAYER_RGGB8: case RIP_FMT_BAYER_RGGB10: case RIP_FMT_BAYER_RGGB12: case RIP_FMT_BAYER_RGGB14: case RIP_FMT_BAYER_RGGB16:
        return launch_fmt<RIP_FMT_BAYER_RGGB8>(s, in, out, W, H, n_frames, to, shift);
    case RIP_FMT_BAYER_BGGR8: case RIP_FMT_BAYER_BGGR10: case RIP_FMT_BAYER_BGGR12: case RIP_FMT_BAYER_BGGR14: case RIP_FMT_BAYER_BGGR16:
        return launch_fmt<RIP_FMT_BAYER_BGGR8>(s, in, out, W, H, n_frames, to, shift);
    case RIP_FMT_BAYER_GRBG8: case RIP_FMT_BAYER_GRBG10: case RIP_FMT_BAYER_GRBG12: case RIP_FMT_BAYER_GRBG14: case RIP_FMT_BAYER_GRBG16:
        return launch_fmt<RIP_FMT_BAYER_GRBG8>(s, in, out, W, H, n_frames, to, shift);
    case RIP_FMT_BAYER_GBRG8: case RIP_FMT_BAYER_GBRG10: case RIP_FMT_BAYER_GBRG12: case RIP_FMT_BAYER_GBRG14: case RIP_FMT_BAYER_GBRG16:
        return launch_fmt<RIP_FMT_BAYER_GBRG8>(s, in, out, W, H, n_frames, to, shift);
    }
    return fail(RIP_EINVAL, "Bayer decode: input format %d is not a Bayer format", in_format);
}

}  // namespace rip
