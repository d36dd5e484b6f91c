// rip_decode.cuh -- the output side of the decode kernels (rip_yuv.cu, rip_bayer.cu): byte packing, the reference's gray of a
// decoded pixel, and the row stores of the six YuvOut targets.  Everything sits in an anonymous namespace, so each
// translation unit that includes it has its own copy of the (r, g) table in constant memory.
#pragma once

#include "rip_common.cuh"
#include "rip_internal.h"

namespace rip {
namespace {

__constant__ uint32_t c_yuv_gray_down[2048] = {
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

// unsaturated R, G, B of one pixel
struct Rgb {
    int r, g, b;
};

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
    return q - ((c_yuv_gray_down[key >> 5] >> (key & 31u)) & 1u);
}

template <int OUT> struct OutFmt;
template <> struct OutFmt<YUV_TO_RGB> { static constexpr int bpp = 3; };
template <> struct OutFmt<YUV_TO_BGR> { static constexpr int bpp = 3; };
template <> struct OutFmt<YUV_TO_RGBA> { static constexpr int bpp = 4; };
template <> struct OutFmt<YUV_TO_BGRA> { static constexpr int bpp = 4; };
template <> struct OutFmt<YUV_TO_GRAY> { static constexpr int bpp = 1; };
template <> struct OutFmt<YUV_TO_GRAY_RGBA> { static constexpr int bpp = 4; };

// the output bytes of one pixel; bpp bytes, low byte first
template <int OUT>
__device__ __forceinline__ uint32_t pixel_word(const Rgb &p)
{
    if constexpr (OUT == YUV_TO_RGBA) return pack4(p.r, p.g, p.b, 255);
    else if constexpr (OUT == YUV_TO_BGRA) return pack4(p.b, p.g, p.r, 255);
    else if constexpr (OUT == YUV_TO_GRAY) return gray_of(pack4(p.r, p.g, p.b, 0));
    else if constexpr (OUT == YUV_TO_GRAY_RGBA) return gray_of(pack4(p.r, p.g, p.b, 0)) * 0x010101u | 0xff000000u;
    else if constexpr (OUT == YUV_TO_RGB) return pack4(p.r, p.g, p.b, 0);
    else return pack4(p.b, p.g, p.r, 0);
}

// the eight pixels to o: 8-byte aligned (16-byte for 4 bytes per pixel)
template <int OUT>
__device__ __forceinline__ void store_x8(uint8_t *o, const uint32_t px[8])
{
    if constexpr (OutFmt<OUT>::bpp == 4) {
        reinterpret_cast<uint4 *>(o)[0] = make_uint4(px[0], px[1], px[2], px[3]);
        reinterpret_cast<uint4 *>(o)[1] = make_uint4(px[4], px[5], px[6], px[7]);
    } else if constexpr (OutFmt<OUT>::bpp == 1) {
        *reinterpret_cast<uint2 *>(o) = make_uint2(pack4(px[0], px[1], px[2], px[3]), pack4(px[4], px[5], px[6], px[7]));
    } else {   // 24 bytes: the 3-byte pixels back to back
        uint2 *o2 = reinterpret_cast<uint2 *>(o);
        o2[0] = make_uint2(px[0] | px[1] << 24, px[1] >> 8 | px[2] << 16);
        o2[1] = make_uint2(px[2] >> 16 | px[3] << 8, px[4] | px[5] << 24);
        o2[2] = make_uint2(px[5] >> 8 | px[6] << 16, px[6] >> 16 | px[7] << 8);
    }
}

template <int OUT>
__device__ __forceinline__ void store_px(uint8_t *o, uint32_t v)
{
#pragma unroll
    for (int b = 0; b < OutFmt<OUT>::bpp; b++) o[b] = (uint8_t)(v >> (8 * b));
}

}  // namespace
}  // namespace rip
