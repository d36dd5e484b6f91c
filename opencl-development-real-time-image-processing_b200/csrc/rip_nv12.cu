// rip_nv12.cu -- NV12 camera frames (RIP_FMT_NV12_COLOR) decoded to colour, or straight to the reference's gray.
//
// Colour is OpenCV's cvtColor(COLOR_YUV2RGB_NV12): BT.601 limited range in 20-bit fixed point, one U,V pair per 2x2
// block of luma:
//     y = max(0, Y - 16) * 1220542,  u = U - 128,  v = V - 128
//     R = sat8((y + 1673527 v + 2^19) >> 20),  G = sat8((y - 852492 v - 409993 u + 2^19) >> 20),  B = sat8((y + 2116026 u + 2^19) >> 20)
// Gray is the reference's (uchar)(0.299 r + 0.587 g + 0.114 b) (Comparator.cpp:41) of the decoded colour.  It does not
// call gray_exact(): neutral chroma (U = V = 128, common in real video) gives r = g = b on every pixel, the case where
// gray_exact replays the double expression.  The exact multiples of 1000 instead take one bit of the (r, g) table that
// the fused kernel uses too (rip_gray_table.inc), and the division by 1000 is the fused kernel's float multiply.
//
// One thread owns two luma rows x 8 columns and the 8 chroma bytes between them, so each U,V pair is loaded once for
// its 2x2 block.  Rows of a width divisible by 8 are read with 64-bit loads and written with 64-bit (1 and 3 bytes per
// pixel) or 128-bit (4 bytes per pixel) stores; saturation and packing are one cvt.pack.sat per two bytes
// (I2IP.U8.S32.SAT).  Other even widths and unaligned buffers take a byte-granular kernel with one 2x2 block per
// thread.  Frames ride in gridDim.y.  Memory-bound by intent: 1.5 bytes per pixel in, 1..4 out.
#include "rip_common.cuh"
#include "rip_internal.h"

namespace rip {
namespace {

__constant__ uint32_t c_nv12_gray_down[2048] = {
#include "rip_gray_table.inc"
};

// d = (c & 0xffff) << 16 | sat_u8(a) << 8 | sat_u8(b)
__device__ __forceinline__ uint32_t i2ip(int a, int b, uint32_t c)
{
    uint32_t d;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// bytes b0..b3 (low to high), each saturated to [0, 255]
__device__ __forceinline__ uint32_t pack4(int b0, int b1, int b2, int b3) { return i2ip(b1, b0, i2ip(b3, b2, 0u)); }
__device__ __forceinline__ uint32_t pack4(uint32_t b0, uint32_t b1, uint32_t b2, uint32_t b3) { return pack4((int)b0, (int)b1, (int)b2, (int)b3); }

struct Chroma {
    int r, g, b;   // chroma part of each channel, with the rounding constant
};

__device__ __forceinline__ Chroma chroma_of(uint32_t U, uint32_t V)
{
    const int u = (int)U - 128, v = (int)V - 128;
    return {(1 << 19) + 1673527 * v, (1 << 19) - 852492 * v - 409993 * u, (1 << 19) + 2116026 * u};
}

// unsaturated R, G, B of one pixel (the >> is arithmetic, as in OpenCV)
struct Rgb {
    int r, g, b;
};

// Y16 = max(Y - 16, 0), already subtracted (four at a time, __vsubus4)
__device__ __forceinline__ Rgb decode(uint32_t Y16, const Chroma &c)
{
    const int y = (int)Y16 * 1220542;
    return {(y + c.r) >> 20, (y + c.g) >> 20, (y + c.b) >> 20};
}

constexpr float kInvK_up = 1.0000000474974513e-3f;   // 0x3A83126F: the float just ABOVE 1/1000
constexpr float kInvK_dn = 9.9999993108212948e-4f;   // 0x3A83126E: the float just BELOW 1/1000

// The reference's gray of a decoded pixel, from its saturated bytes (r, g, b, 0).  t = 299 r + 587 g + 114 b by two IDP.2A;
// floor(t / 1000) as in the fused kernel: t's bit pattern read as a float is the denormal t * 2^-149, one multiply rounded
// toward -inf by the float just above 1/1000 leaves floor(t / 1000) in the bit pattern, and a multiply-add rounded toward +inf
// with the float just below 1/1000 is 1 exactly when t is a nonzero multiple of 1000 (rip_debug_selftest checks the same
// arithmetic on all 2^24 triples).  Only there can the reference's double expression land one below t / 1000, as the (r, g)
// table bit says.
__device__ __forceinline__ uint32_t gray_of(uint32_t rgb0)
{
    const uint32_t t = __dp2a_hi(114u, rgb0, __dp2a_lo(299u | (587u << 16), rgb0, 0u));
    const float tf = __uint_as_float(t);
    const uint32_t q = __float_as_uint(__fmul_rd(tf, kInvK_up));
    if (__float_as_uint(__fmaf_ru(tf, -kInvK_dn, __uint_as_float(q))) != 1u) return q;
    const uint32_t key = rgb0 & 0xffffu;
    return q - ((c_nv12_gray_down[key >> 5] >> (key & 31u)) & 1u);
}

template <int OUT> struct OutFmt;
template <> struct OutFmt<NV12_TO_RGB> { static constexpr int bpp = 3; };
template <> struct OutFmt<NV12_TO_BGR> { static constexpr int bpp = 3; };
template <> struct OutFmt<NV12_TO_RGBA> { static constexpr int bpp = 4; };
template <> struct OutFmt<NV12_TO_BGRA> { static constexpr int bpp = 4; };
template <> struct OutFmt<NV12_TO_GRAY> { static constexpr int bpp = 1; };
template <> struct OutFmt<NV12_TO_GRAY_RGBA> { static constexpr int bpp = 4; };

// the output bytes of one pixel; bpp bytes, low byte first
template <int OUT>
__device__ __forceinline__ uint32_t pixel_word(const Rgb &p)
{
    if constexpr (OUT == NV12_TO_RGBA) return pack4(p.r, p.g, p.b, 255);
    else if constexpr (OUT == NV12_TO_BGRA) return pack4(p.b, p.g, p.r, 255);
    else if constexpr (OUT == NV12_TO_GRAY) return gray_of(pack4(p.r, p.g, p.b, 0));
    else if constexpr (OUT == NV12_TO_GRAY_RGBA) return gray_of(pack4(p.r, p.g, p.b, 0)) * 0x010101u | 0xff000000u;
    else if constexpr (OUT == NV12_TO_RGB) return pack4(p.r, p.g, p.b, 0);
    else return pack4(p.b, p.g, p.r, 0);
}

// W % 8 == 0, input 8-byte aligned, output 8-byte (16-byte for 4 bytes per pixel) aligned
template <int OUT>
__global__ void __launch_bounds__(256)
nv12_kernel_x8(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int W, int H, int f0)
{
    constexpr int BPP = OutFmt<OUT>::bpp;
    const int cols = W >> 3;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    const int rp = u / cols, c = u - rp * cols;   // row pair, 8-column group
    if (rp >= (H >> 1)) return;
    const size_t f = (size_t)f0 + blockIdx.y;
    const uint8_t *luma = in + f * ((size_t)W * H * 3 / 2) + (size_t)(2 * rp) * W + 8 * c;
    const uint8_t *uv = in + f * ((size_t)W * H * 3 / 2) + (size_t)W * H + (size_t)rp * W + 8 * c;
    const uint2 y0 = __ldg(reinterpret_cast<const uint2 *>(luma));
    const uint2 y1 = __ldg(reinterpret_cast<const uint2 *>(luma + W));
    const uint2 cv = __ldg(reinterpret_cast<const uint2 *>(uv));
    const uint32_t Y[2][2] = {{__vsubus4(y0.x, 0x10101010u), __vsubus4(y0.y, 0x10101010u)},
                              {__vsubus4(y1.x, 0x10101010u), __vsubus4(y1.y, 0x10101010u)}};   // max(Y - 16, 0)
    const uint32_t UV[2] = {cv.x, cv.y};
    uint8_t *orow = out + (f * H * W + (size_t)(2 * rp) * W + 8 * c) * BPP;
#pragma unroll
    for (int row = 0; row < 2; row++) {
        uint32_t px[8];
#pragma unroll
        for (int k = 0; k < 4; k++) {   // chroma pair k serves columns 2k and 2k+1
            const uint32_t w = UV[k >> 1], s = 16 * (k & 1);
            const Chroma ch = chroma_of((w >> s) & 0xffu, (w >> (s + 8)) & 0xffu);
            const uint32_t yw = Y[row][k >> 1];
            px[2 * k] = pixel_word<OUT>(decode((yw >> s) & 0xffu, ch));
            px[2 * k + 1] = pixel_word<OUT>(decode((yw >> (s + 8)) & 0xffu, ch));
        }
        uint8_t *o = orow + (size_t)row * W * BPP;
        if constexpr (BPP == 4) {
            reinterpret_cast<uint4 *>(o)[0] = make_uint4(px[0], px[1], px[2], px[3]);
            reinterpret_cast<uint4 *>(o)[1] = make_uint4(px[4], px[5], px[6], px[7]);
        } else if constexpr (BPP == 1) {
            *reinterpret_cast<uint2 *>(o) = make_uint2(pack4(px[0], px[1], px[2], px[3]), pack4(px[4], px[5], px[6], px[7]));
        } else {   // 24 bytes: the 3-byte pixels back to back
            uint2 *o2 = reinterpret_cast<uint2 *>(o);
            o2[0] = make_uint2(px[0] | px[1] << 24, px[1] >> 8 | px[2] << 16);
            o2[1] = make_uint2(px[2] >> 16 | px[3] << 8, px[4] | px[5] << 24);
            o2[2] = make_uint2(px[5] >> 8 | px[6] << 16, px[6] >> 16 | px[7] << 8);
        }
    }
}

// any even width, any alignment: one 2x2 block per thread, byte loads and stores
template <int OUT>
__global__ void __launch_bounds__(256)
nv12_kernel_x2(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int W, int H, int f0)
{
    constexpr int BPP = OutFmt<OUT>::bpp;
    const int cols = W >> 1;
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    const int rp = u / cols, c = u - rp * cols;
    if (rp >= (H >> 1)) return;
    const size_t f = (size_t)f0 + blockIdx.y;
    const uint8_t *luma = in + f * ((size_t)W * H * 3 / 2) + (size_t)(2 * rp) * W + 2 * c;
    const uint8_t *uv = in + f * ((size_t)W * H * 3 / 2) + (size_t)W * H + (size_t)rp * W + 2 * c;
    const Chroma ch = chroma_of(__ldg(uv), __ldg(uv + 1));
#pragma unroll
    for (int row = 0; row < 2; row++) {
        uint8_t *o = out + (f * H * W + (size_t)(2 * rp + row) * W + 2 * c) * BPP;
#pragma unroll
        for (int i = 0; i < 2; i++) {
            const uint32_t v = pixel_word<OUT>(decode(max((int)__ldg(luma + (size_t)row * W + i) - 16, 0), ch));
#pragma unroll
            for (int b = 0; b < BPP; b++) o[i * BPP + b] = (uint8_t)(v >> (8 * b));
        }
    }
}

template <int OUT>
int launch_t(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames)
{
    constexpr int BPP = OutFmt<OUT>::bpp;
    const uintptr_t out_align = BPP == 4 ? 15u : 7u;
    const bool x8 = (W & 7) == 0 && (reinterpret_cast<uintptr_t>(in) & 7u) == 0 && (reinterpret_cast<uintptr_t>(out) & out_align) == 0;
    const long long units = (long long)(H / 2) * (x8 ? W / 8 : W / 2);   // threads per frame
    const dim3 block(256);
    for (int f0 = 0; f0 < n_frames; f0 += 65535) {
        const dim3 grid((unsigned)((units + 255) / 256), (unsigned)min(n_frames - f0, 65535));
        if (x8) nv12_kernel_x8<OUT><<<grid, block, 0, s>>>(in, out, W, H, f0);
        else nv12_kernel_x2<OUT><<<grid, block, 0, s>>>(in, out, W, H, f0);
        RIP_LAUNCH_CHECK();
    }
    return RIP_OK;
}

}  // namespace

int launch_nv12(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames, Nv12Out to)
{
    if ((W & 1) || (H & 1)) return fail(RIP_EINVAL, "NV12 frames need an even width and height (got %d x %d)", W, H);
    if ((long long)(H / 2) * (W / 2) > 0x7fffff00ll)   // (thread indices are 32-bit)
        return fail(RIP_EINVAL, "NV12 frame of %d x %d is too large", W, H);
    switch (to) {
    case NV12_TO_RGB: return launch_t<NV12_TO_RGB>(s, in, out, W, H, n_frames);
    case NV12_TO_BGR: return launch_t<NV12_TO_BGR>(s, in, out, W, H, n_frames);
    case NV12_TO_RGBA: return launch_t<NV12_TO_RGBA>(s, in, out, W, H, n_frames);
    case NV12_TO_BGRA: return launch_t<NV12_TO_BGRA>(s, in, out, W, H, n_frames);
    case NV12_TO_GRAY: return launch_t<NV12_TO_GRAY>(s, in, out, W, H, n_frames);
    case NV12_TO_GRAY_RGBA: return launch_t<NV12_TO_GRAY_RGBA>(s, in, out, W, H, n_frames);
    }
    return fail(RIP_EINVAL, "NV12 decode: bad output %d", (int)to);
}

}  // namespace rip
