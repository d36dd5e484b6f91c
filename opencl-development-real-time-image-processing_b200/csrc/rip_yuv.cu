// rip_yuv.cu -- camera frames (RIP_FMT_NV12_COLOR, RIP_FMT_I420, RIP_FMT_YUYV, RIP_FMT_UYVY) decoded to colour, or straight
// to the reference's gray.  launch_yuv is also the entry for the Bayer formats, whose kernels are in rip_bayer.cu; the
// output side of both (packing, gray, stores) is rip_decode.cuh.
//
// Colour is OpenCV's cvtColor(COLOR_YUV2RGB_NV12 / _I420 / _YUYV / _UYVY): BT.601 limited range in 20-bit fixed point.  The
// four layouts differ only in where Y, U and V sit (one U,V pair per 2x2 block of luma for NV12 and I420, per horizontal
// pixel pair for YUYV and UYVY); every pixel then goes through the same arithmetic:
//     y = max(0, Y - 16) * 1220542,  u = U - 128,  v = V - 128
//     R = sat8((y + 1673527 v + 2^19) >> 20),  G = sat8((y - 852492 v - 409993 u + 2^19) >> 20),  B = sat8((y + 2116026 u + 2^19) >> 20)
// Gray is the reference's (uchar)(0.299 r + 0.587 g + 0.114 b) (Comparator.cpp:41) of the decoded colour.  It does not
// call gray_exact(): neutral chroma (U = V = 128, common in real video) gives r = g = b on every pixel, the case where
// gray_exact replays the double expression.  The exact multiples of 1000 instead take one bit of the (r, g) table that
// the fused kernel uses too (rip_gray_table.inc), and the division by 1000 is the fused kernel's float multiply.
//
// 4:2:0 (NV12, I420): one thread owns two luma rows x 8 columns and the 8 chroma bytes between them, so each U,V pair is
// loaded once for its 2x2 block: one 64-bit word of NV12's interleaved plane, or one 32-bit word of each I420 plane.
// 4:2:2 (YUYV, UYVY): one thread owns 8 pixels of one row, one 16-byte load, rearranged into the same luma and chroma words.
// Rows are written with 64-bit (1 and 3 bytes per pixel) or 128-bit (4 bytes per pixel) stores; saturation and packing are
// one cvt.pack.sat per two bytes (I2IP.U8.S32.SAT).  Widths that are not a multiple of 8 and unaligned buffers take
// byte-granular kernels (one 2x2 block, or one pixel pair, per thread).  Frames ride in gridDim.y.  Memory-bound by intent:
// 1.5 (4:2:0) or 2 (4:2:2) bytes per pixel in, 1..4 out.
#include "rip_decode.cuh"

namespace rip {
namespace {

struct Chroma {
    int r, g, b;   // chroma part of each channel, with the rounding constant
};

__device__ __forceinline__ Chroma chroma_of(uint32_t U, uint32_t V)
{
    const int u = (int)U - 128, v = (int)V - 128;
    return {(1 << 19) + 1673527 * v, (1 << 19) - 852492 * v - 409993 * u, (1 << 19) + 2116026 * u};
}

// Y16 = max(Y - 16, 0), already subtracted (four at a time, __vsubus4)
__device__ __forceinline__ Rgb decode(uint32_t Y16, const Chroma &c)
{
    const int y = (int)Y16 * 1220542;
    return {(y + c.r) >> 20, (y + c.g) >> 20, (y + c.b) >> 20};
}

// Eight pixels of one row.  Y: max(Y - 16, 0) of pixels 0..3 and 4..7, low byte first; UV: the U,V byte pairs (U low)
// serving pixels 0,1 and 2,3, then 4,5 and 6,7.
template <int OUT>
__device__ __forceinline__ void row_x8(uint32_t px[8], const uint32_t Y[2], const uint32_t UV[2])
{
#pragma unroll
    for (int k = 0; k < 4; k++) {   // chroma pair k serves columns 2k and 2k+1
        const uint32_t w = UV[k >> 1], s = 16 * (k & 1);
        const Chroma ch = chroma_of((w >> s) & 0xffu, (w >> (s + 8)) & 0xffu);
        const uint32_t yw = Y[k >> 1];
        px[2 * k] = pixel_word<OUT>(decode((yw >> s) & 0xffu, ch));
        px[2 * k + 1] = pixel_word<OUT>(decode((yw >> (s + 8)) & 0xffu, ch));
    }
}

// one pixel of luma Y (not yet reduced by 16)
template <int OUT>
__device__ __forceinline__ uint32_t pixel_of(uint32_t Y, const Chroma &ch) { return pixel_word<OUT>(decode(max((int)Y - 16, 0), ch)); }

// 4:2:0 chroma of frame f, after its W*H luma plane: NV12 interleaves U,V in one plane of W bytes per row; I420 keeps a U
// plane and then a V plane, each of W/2 bytes per row and (W/2) * (H/2) bytes.  chroma_at is the U byte of pair `pair` of
// chroma row rp; the V byte is v_offset further.
template <bool I420>
__device__ __forceinline__ const uint8_t *chroma_at(const uint8_t *in, size_t f, int W, int H, int rp, int pair)
{
    if constexpr (I420) return in + f * ((size_t)W * H * 3 / 2) + (size_t)W * H + (size_t)rp * (W >> 1) + pair;
    else return in + f * ((size_t)W * H * 3 / 2) + (size_t)W * H + (size_t)rp * W + 2 * pair;
}

template <bool I420>
__device__ __forceinline__ size_t v_offset(int W, int H) { return I420 ? (size_t)(W >> 1) * (H >> 1) : 1; }

// 4:2:0, W % 8 == 0, input 8-byte aligned, output 8-byte (16-byte for 4 bytes per pixel) aligned
template <int OUT, bool I420>
__global__ void __launch_bounds__(256)
yuv420_kernel_x8(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int W, int H, int f0)
{
    constexpr int BPP = OutFmt<OUT>::bpp;
    const int cols = W >> 3;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    const int rp = u / cols, c = u - rp * cols;   // row pair, 8-column group
    if (rp >= (H >> 1)) return;
    const size_t f = (size_t)f0 + blockIdx.y;
    const uint8_t *luma = in + f * ((size_t)W * H * 3 / 2) + (size_t)(2 * rp) * W + 8 * c;
    const uint8_t *uv = chroma_at<I420>(in, f, W, H, rp, 4 * c);   // 8-byte aligned (NV12), 4-byte (I420)
    const uint2 y0 = __ldg(reinterpret_cast<const uint2 *>(luma));
    const uint2 y1 = __ldg(reinterpret_cast<const uint2 *>(luma + W));
    uint2 cv;
    if constexpr (I420) {   // u0 u1 u2 u3 and v0 v1 v2 v3 to u0 v0 u1 v1, u2 v2 u3 v3
        const uint32_t U = __ldg(reinterpret_cast<const uint32_t *>(uv));
        const uint32_t V = __ldg(reinterpret_cast<const uint32_t *>(uv + v_offset<I420>(W, H)));
        cv = make_uint2(__byte_perm(U, V, 0x5140), __byte_perm(U, V, 0x7362));
    } else {
        cv = __ldg(reinterpret_cast<const uint2 *>(uv));
    }
    const uint32_t Y[2][2] = {{__vsubus4(y0.x, 0x10101010u), __vsubus4(y0.y, 0x10101010u)},
                              {__vsubus4(y1.x, 0x10101010u), __vsubus4(y1.y, 0x10101010u)}};   // max(Y - 16, 0)
    const uint32_t UV[2] = {cv.x, cv.y};
    uint8_t *orow = out + (f * H * W + (size_t)(2 * rp) * W + 8 * c) * BPP;
#pragma unroll
    for (int row = 0; row < 2; row++) {
        uint32_t px[8];
        row_x8<OUT>(px, Y[row], UV);
        store_x8<OUT>(orow + (size_t)row * W * BPP, px);
    }
}

// 4:2:0, any even width, any alignment: one 2x2 block per thread, byte loads and stores
template <int OUT, bool I420>
__global__ void __launch_bounds__(256)
yuv420_kernel_x2(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int W, int H, int f0)
{
    constexpr int BPP = OutFmt<OUT>::bpp;
    const int cols = W >> 1;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    const int rp = u / cols, c = u - rp * cols;
    if (rp >= (H >> 1)) return;
    const size_t f = (size_t)f0 + blockIdx.y;
    const uint8_t *luma = in + f * ((size_t)W * H * 3 / 2) + (size_t)(2 * rp) * W + 2 * c;
    const uint8_t *uv = chroma_at<I420>(in, f, W, H, rp, c);
    const Chroma ch = chroma_of(__ldg(uv), __ldg(uv + v_offset<I420>(W, H)));
#pragma unroll
    for (int row = 0; row < 2; row++) {
        uint8_t *o = out + (f * H * W + (size_t)(2 * rp + row) * W + 2 * c) * BPP;
#pragma unroll
        for (int i = 0; i < 2; i++) {
            const uint32_t v = pixel_of<OUT>(__ldg(luma + (size_t)row * W + i), ch);
            store_px<OUT>(o + i * BPP, v);
        }
    }
}

// 4:2:2 byte positions in a 4-byte pixel pair: YUYV is Y0 U Y1 V, UYVY is U Y0 V Y1.  ysel / uvsel: the __byte_perm
// selectors that gather the luma bytes, or the U,V pairs, of two pixel pairs into one word.
template <bool UYVY> struct Packed422 {
    static constexpr int y0 = UYVY ? 1 : 0, u = UYVY ? 0 : 1, v = UYVY ? 2 : 3;
    static constexpr uint32_t ysel = UYVY ? 0x7531u : 0x6420u, uvsel = UYVY ? 0x6420u : 0x7531u;
};

// 4:2:2, W % 8 == 0, input 16-byte aligned, output as for 4:2:0: 8 pixels of one row per thread
template <int OUT, bool UYVY>
__global__ void __launch_bounds__(256)
yuv422_kernel_x8(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int W, int H, int f0)
{
    using P = Packed422<UYVY>;
    const int cols = W >> 3;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = u / cols, c = u - r * cols;   // row, 8-column group
    if (r >= H) return;
    const size_t row = ((size_t)f0 + blockIdx.y) * H + r;   // row of the whole batch
    const uint4 q = __ldg(reinterpret_cast<const uint4 *>(in + row * 2 * W + 16 * c));
    const uint32_t Y[2] = {__vsubus4(__byte_perm(q.x, q.y, P::ysel), 0x10101010u), __vsubus4(__byte_perm(q.z, q.w, P::ysel), 0x10101010u)};
    const uint32_t UV[2] = {__byte_perm(q.x, q.y, P::uvsel), __byte_perm(q.z, q.w, P::uvsel)};
    uint32_t px[8];
    row_x8<OUT>(px, Y, UV);
    store_x8<OUT>(out + (row * W + 8 * c) * OutFmt<OUT>::bpp, px);
}

// 4:2:2, any even width, any height, any alignment: one pixel pair per thread, byte loads and stores
template <int OUT, bool UYVY>
__global__ void __launch_bounds__(256)
yuv422_kernel_x2(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int W, int H, int f0)
{
    using P = Packed422<UYVY>;
    constexpr int BPP = OutFmt<OUT>::bpp;
    const int cols = W >> 1;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = u / cols, c = u - r * cols;
    if (r >= H) return;
    const size_t row = ((size_t)f0 + blockIdx.y) * H + r;
    const uint8_t *p = in + row * 2 * W + 4 * c;
    const Chroma ch = chroma_of(__ldg(p + P::u), __ldg(p + P::v));
    uint8_t *o = out + (row * W + 2 * c) * BPP;
    store_px<OUT>(o, pixel_of<OUT>(__ldg(p + P::y0), ch));
    store_px<OUT>(o + BPP, pixel_of<OUT>(__ldg(p + P::y0 + 2), ch));
}

template <int OUT, int FMT>
int launch_t(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames)
{
    constexpr int BPP = OutFmt<OUT>::bpp;
    constexpr bool packed = FMT == RIP_FMT_YUYV || FMT == RIP_FMT_UYVY;   // 4:2:2: a thread per row; 4:2:0: per row pair
    const uintptr_t in_align = packed ? 15u : 7u, out_align = BPP == 4 ? 15u : 7u;
    const bool x8 = (W & 7) == 0 && (reinterpret_cast<uintptr_t>(in) & in_align) == 0 && (reinterpret_cast<uintptr_t>(out) & out_align) == 0;
    const long long units = (long long)(packed ? H : H / 2) * (x8 ? W / 8 : W / 2);   // threads per frame
    const dim3 block(256);
    for (int f0 = 0; f0 < n_frames; f0 += 65535) {
        const dim3 grid((unsigned)((units + 255) / 256), (unsigned)min(n_frames - f0, 65535));
        if constexpr (packed) {
            if (x8) yuv422_kernel_x8<OUT, FMT == RIP_FMT_UYVY><<<grid, block, 0, s>>>(in, out, W, H, f0);
            else yuv422_kernel_x2<OUT, FMT == RIP_FMT_UYVY><<<grid, block, 0, s>>>(in, out, W, H, f0);
        } else {
            if (x8) yuv420_kernel_x8<OUT, FMT == RIP_FMT_I420><<<grid, block, 0, s>>>(in, out, W, H, f0);
            else yuv420_kernel_x2<OUT, FMT == RIP_FMT_I420><<<grid, block, 0, s>>>(in, out, W, H, f0);
        }
        RIP_LAUNCH_CHECK();
    }
    return RIP_OK;
}

template <int FMT>
int launch_fmt(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames, YuvOut to)
{
    switch (to) {
    case YUV_TO_RGB: return launch_t<YUV_TO_RGB, FMT>(s, in, out, W, H, n_frames);
    case YUV_TO_BGR: return launch_t<YUV_TO_BGR, FMT>(s, in, out, W, H, n_frames);
    case YUV_TO_RGBA: return launch_t<YUV_TO_RGBA, FMT>(s, in, out, W, H, n_frames);
    case YUV_TO_BGRA: return launch_t<YUV_TO_BGRA, FMT>(s, in, out, W, H, n_frames);
    case YUV_TO_GRAY: return launch_t<YUV_TO_GRAY, FMT>(s, in, out, W, H, n_frames);
    case YUV_TO_GRAY_RGBA: return launch_t<YUV_TO_GRAY_RGBA, FMT>(s, in, out, W, H, n_frames);
    }
    return fail(RIP_EINVAL, "YUV decode: bad output %d", (int)to);
}

}  // namespace

int check_yuv_shape(int fmt, int W, int H)
{
    if (!decodes_to_color(fmt)) return fail(RIP_EINVAL, "YUV decode: input format %d is not decoded to colour", fmt);
    const Format &f = *format_of(fmt);
    if (!shape_ok(f, W, H)) {
        if (f.packing == BAYER_GENICAM)
            return fail(RIP_EINVAL, "%s frames need a width that is a multiple of %d and at least 4, and a height of at least 3 "
                        "(got %d x %d): rows are W*%d/8 bytes with no padding, and a width that is not a multiple of %d "
                        "would start rows inside a byte", f.name, f.w_mul, W, H, f.bits, f.w_mul);
        if (f.packing == BAYER_MIPI)
            return fail(RIP_EINVAL, "%s frames need a width that is a multiple of %d and at least 4, and a height of at least 3 "
                        "(got %d x %d): rows are W*%d/8 bytes with no padding", f.name, f.w_mul, W, H, f.bits);
        if (f.layout == LAYOUT_BAYER)
            return fail(RIP_EINVAL, "%s frames need a width and height of at least 3 (got %d x %d)", f.name, W, H);
        if (f.layout == LAYOUT_YUV422) return fail(RIP_EINVAL, "%s frames need an even width (got %d x %d)", f.name, W, H);
        return fail(RIP_EINVAL, "%s frames need an even width and height (got %d x %d)", f.name, W, H);
    }
    // threads of the x1 / x2 kernels per frame: one per Bayer pixel, 4:2:2 pixel pair or 4:2:0 2x2 block
    const long long units = f.layout == LAYOUT_BAYER ? (long long)W * H : (long long)(H / f.h_mul) * (W / f.w_mul);
    if (units > 0x7fffff00ll)   // (thread indices are 32-bit)
        return fail(RIP_EINVAL, "%s frame of %d x %d is too large", f.name, W, H);
    return RIP_OK;
}

int launch_yuv(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames, int in_format, YuvOut to)
{
    if (int rc = check_yuv_shape(in_format, W, H)) return rc;
    if (format_of(in_format)->layout == LAYOUT_BAYER) return launch_bayer(s, in, out, W, H, n_frames, in_format, to);
    switch (in_format) {
    case RIP_FMT_NV12_COLOR: return launch_fmt<RIP_FMT_NV12_COLOR>(s, in, out, W, H, n_frames, to);
    case RIP_FMT_I420: return launch_fmt<RIP_FMT_I420>(s, in, out, W, H, n_frames, to);
    case RIP_FMT_YUYV: return launch_fmt<RIP_FMT_YUYV>(s, in, out, W, H, n_frames, to);
    default: return launch_fmt<RIP_FMT_UYVY>(s, in, out, W, H, n_frames, to);
    }
}

}  // namespace rip
