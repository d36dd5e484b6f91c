// rip_formats.h -- every pixel format of include/rip_cuda.h described once: its name, how its bytes are laid out, its bytes
// per frame and the shapes it accepts.  The library's format and shape checks, frame strides and Bayer kernel routing, and the
// C++ Controller's input sizes, read these rows, so a new format is one row here plus its kernels.  Plain C++17 (no CUDA),
// read by librip_cuda.so and librip_host.so alike.
#pragma once

#include <stddef.h>

#include "rip_cuda.h"

namespace rip {

enum FormatLayout {
    LAYOUT_INTERLEAVED,   // GRAY8, RGB8, BGR8, RGBA8, BGRA8: used as is
    LAYOUT_NV12_LUMA,     // NV12: the W*H luma plane is the gray image; the chroma plane behind it is never read
    LAYOUT_YUV420,        // NV12_COLOR, I420: decoded to colour, one U,V pair per 2x2 block
    LAYOUT_YUV422,        // YUYV, UYVY: decoded to colour, one U,V pair per horizontal pixel pair
    LAYOUT_BAYER,         // Bayer raw frames: demosaiced to colour
};

// how a Bayer format stores its samples: whole bytes or 16-bit words, MIPI CSI-2 RAW10 / RAW12, or a GenICam bit stream
enum BayerPacking { BAYER_UNPACKED, BAYER_MIPI, BAYER_GENICAM };

struct Format {
    int code;                         // RIP_FMT_*
    const char *name;                 // the code's name without the RIP_FMT_ prefix
    FormatLayout layout;
    int channels;                     // of the image the operations see: 1, 3 or 4 interleaved, 1 for NV12 (its luma plane),
                                      // 3 for the decoded layouts (R, G, B)
    bool bgr;                         // interleaved with blue first
    int pattern;                      // Bayer: 0 RGGB, 1 BGGR, 2 GRBG, 3 GBRG (the order of codes 12-15); -1 otherwise
    int bits;                         // Bayer: bits per sample; 0 otherwise
    BayerPacking packing;
    int bytes_num, bytes_den;         // bytes per frame: W * H * bytes_num / bytes_den
    int w_mul, h_mul, w_min, h_min;   // accepted shapes: W a multiple of w_mul and >= w_min, H of h_mul and >= h_min
};

#define RIP_FORMAT(NAME, ...) Format{RIP_FMT_##NAME, #NAME, __VA_ARGS__}
inline constexpr Format kFormats[] = {
    // name, layout, channels, bgr, pattern, bits, packing, bytes_num, bytes_den, w_mul, h_mul, w_min, h_min
    RIP_FORMAT(GRAY8,                 LAYOUT_INTERLEAVED, 1, false, -1,  0, BAYER_UNPACKED, 1, 1,  1, 1, 1, 1),
    RIP_FORMAT(RGB8,                  LAYOUT_INTERLEAVED, 3, false, -1,  0, BAYER_UNPACKED, 3, 1,  1, 1, 1, 1),
    RIP_FORMAT(RGBA8,                 LAYOUT_INTERLEAVED, 4, false, -1,  0, BAYER_UNPACKED, 4, 1,  1, 1, 1, 1),
    RIP_FORMAT(BGR8,                  LAYOUT_INTERLEAVED, 3, true,  -1,  0, BAYER_UNPACKED, 3, 1,  1, 1, 1, 1),
    RIP_FORMAT(BGRA8,                 LAYOUT_INTERLEAVED, 4, true,  -1,  0, BAYER_UNPACKED, 4, 1,  1, 1, 1, 1),
    RIP_FORMAT(NV12,                  LAYOUT_NV12_LUMA,   1, false, -1,  0, BAYER_UNPACKED, 3, 2,  1, 2, 1, 1),
    RIP_FORMAT(NV12_COLOR,            LAYOUT_YUV420,      3, false, -1,  0, BAYER_UNPACKED, 3, 2,  2, 2, 1, 1),
    RIP_FORMAT(YUYV,                  LAYOUT_YUV422,      3, false, -1,  0, BAYER_UNPACKED, 2, 1,  2, 1, 1, 1),
    RIP_FORMAT(UYVY,                  LAYOUT_YUV422,      3, false, -1,  0, BAYER_UNPACKED, 2, 1,  2, 1, 1, 1),
    RIP_FORMAT(I420,                  LAYOUT_YUV420,      3, false, -1,  0, BAYER_UNPACKED, 3, 2,  2, 2, 1, 1),
    RIP_FORMAT(BAYER_RGGB8,           LAYOUT_BAYER,       3, false,  0,  8, BAYER_UNPACKED, 1, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_BGGR8,           LAYOUT_BAYER,       3, false,  1,  8, BAYER_UNPACKED, 1, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_GRBG8,           LAYOUT_BAYER,       3, false,  2,  8, BAYER_UNPACKED, 1, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_GBRG8,           LAYOUT_BAYER,       3, false,  3,  8, BAYER_UNPACKED, 1, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_RGGB10,          LAYOUT_BAYER,       3, false,  0, 10, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_BGGR10,          LAYOUT_BAYER,       3, false,  1, 10, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_GRBG10,          LAYOUT_BAYER,       3, false,  2, 10, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_GBRG10,          LAYOUT_BAYER,       3, false,  3, 10, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_RGGB12,          LAYOUT_BAYER,       3, false,  0, 12, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_BGGR12,          LAYOUT_BAYER,       3, false,  1, 12, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_GRBG12,          LAYOUT_BAYER,       3, false,  2, 12, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_GBRG12,          LAYOUT_BAYER,       3, false,  3, 12, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_RGGB14,          LAYOUT_BAYER,       3, false,  0, 14, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_BGGR14,          LAYOUT_BAYER,       3, false,  1, 14, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_GRBG14,          LAYOUT_BAYER,       3, false,  2, 14, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_GBRG14,          LAYOUT_BAYER,       3, false,  3, 14, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_RGGB16,          LAYOUT_BAYER,       3, false,  0, 16, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_BGGR16,          LAYOUT_BAYER,       3, false,  1, 16, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_GRBG16,          LAYOUT_BAYER,       3, false,  2, 16, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    RIP_FORMAT(BAYER_GBRG16,          LAYOUT_BAYER,       3, false,  3, 16, BAYER_UNPACKED, 2, 1,  1, 1, 3, 3),
    // packed: rows of whole bytes with no padding, so W is a multiple of the pixels in one byte group (4 in 5, or 2 in 3)
    RIP_FORMAT(BAYER_RGGB10P_MIPI,    LAYOUT_BAYER,       3, false,  0, 10, BAYER_MIPI,     5, 4,  4, 1, 4, 3),
    RIP_FORMAT(BAYER_BGGR10P_MIPI,    LAYOUT_BAYER,       3, false,  1, 10, BAYER_MIPI,     5, 4,  4, 1, 4, 3),
    RIP_FORMAT(BAYER_GRBG10P_MIPI,    LAYOUT_BAYER,       3, false,  2, 10, BAYER_MIPI,     5, 4,  4, 1, 4, 3),
    RIP_FORMAT(BAYER_GBRG10P_MIPI,    LAYOUT_BAYER,       3, false,  3, 10, BAYER_MIPI,     5, 4,  4, 1, 4, 3),
    RIP_FORMAT(BAYER_RGGB12P_MIPI,    LAYOUT_BAYER,       3, false,  0, 12, BAYER_MIPI,     3, 2,  2, 1, 4, 3),
    RIP_FORMAT(BAYER_BGGR12P_MIPI,    LAYOUT_BAYER,       3, false,  1, 12, BAYER_MIPI,     3, 2,  2, 1, 4, 3),
    RIP_FORMAT(BAYER_GRBG12P_MIPI,    LAYOUT_BAYER,       3, false,  2, 12, BAYER_MIPI,     3, 2,  2, 1, 4, 3),
    RIP_FORMAT(BAYER_GBRG12P_MIPI,    LAYOUT_BAYER,       3, false,  3, 12, BAYER_MIPI,     3, 2,  2, 1, 4, 3),
    RIP_FORMAT(BAYER_RGGB10P_GENICAM, LAYOUT_BAYER,       3, false,  0, 10, BAYER_GENICAM,  5, 4,  4, 1, 4, 3),
    RIP_FORMAT(BAYER_BGGR10P_GENICAM, LAYOUT_BAYER,       3, false,  1, 10, BAYER_GENICAM,  5, 4,  4, 1, 4, 3),
    RIP_FORMAT(BAYER_GRBG10P_GENICAM, LAYOUT_BAYER,       3, false,  2, 10, BAYER_GENICAM,  5, 4,  4, 1, 4, 3),
    RIP_FORMAT(BAYER_GBRG10P_GENICAM, LAYOUT_BAYER,       3, false,  3, 10, BAYER_GENICAM,  5, 4,  4, 1, 4, 3),
    RIP_FORMAT(BAYER_RGGB12P_GENICAM, LAYOUT_BAYER,       3, false,  0, 12, BAYER_GENICAM,  3, 2,  2, 1, 4, 3),
    RIP_FORMAT(BAYER_BGGR12P_GENICAM, LAYOUT_BAYER,       3, false,  1, 12, BAYER_GENICAM,  3, 2,  2, 1, 4, 3),
    RIP_FORMAT(BAYER_GRBG12P_GENICAM, LAYOUT_BAYER,       3, false,  2, 12, BAYER_GENICAM,  3, 2,  2, 1, 4, 3),
    RIP_FORMAT(BAYER_GBRG12P_GENICAM, LAYOUT_BAYER,       3, false,  3, 12, BAYER_GENICAM,  3, 2,  2, 1, 4, 3),
};
#undef RIP_FORMAT

// the row of format code `fmt`, or nullptr for a code include/rip_cuda.h does not define
inline const Format *format_of(int fmt)
{
    for (const Format &f : kFormats)
        if (f.code == fmt) return &f;
    return nullptr;
}

// NV12_COLOR, YUYV, UYVY, I420 and Bayer: decoded to colour before any operation
inline bool decodes_to_color(int fmt)
{
    const Format *f = format_of(fmt);
    return f && f->layout != LAYOUT_INTERLEAVED && f->layout != LAYOUT_NV12_LUMA;
}

// W and H positive
inline bool shape_ok(const Format &f, int W, int H) { return W >= f.w_min && H >= f.h_min && W % f.w_mul == 0 && H % f.h_mul == 0; }

// bytes from one whole frame of a batch to the next
inline size_t frame_bytes(const Format &f, int W, int H) { return (size_t)W * H * f.bytes_num / f.bytes_den; }

}  // namespace rip
