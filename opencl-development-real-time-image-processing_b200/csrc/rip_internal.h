// rip_internal.h -- launchers shared between the translation units of librip_cuda.so (not exported).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "rip_common.cuh"

namespace rip {

// rip_stages.cu
int launch_gray(cudaStream_t s, const uint8_t *in, uint8_t *out, long long npx, int fmt, int out_mode, int device);
// KxK Gaussian: the separable guard-band kernel (rip_blur_sep.cu) when the weights allow it, else the plain
// reference-order kernel (rip_stages.cu); both bit-exact
int launch_blur(cudaStream_t s, const uint8_t *src, uint8_t *dst, int W, int H, int n_frames, int cn,
                int ksize, const Weights &wts, int src_row0, int src_rows, int out_row0, int out_rows);
int launch_blur_exact(cudaStream_t s, const uint8_t *src, uint8_t *dst, int W, int H, int n_frames, int cn,
                      int ksize, const Weights &wts, int src_row0, int src_rows, int out_row0, int out_rows);
// rip_blur_sep.cu; RIP_EUNSUPPORTED (no error recorded) = use the exact kernel
int launch_blur_sep(cudaStream_t s, const uint8_t *src, uint8_t *dst, int W, int H, int n_frames, int cn,
                    int ksize, const Weights &wts, int src_row0, int src_rows, int out_row0, int out_rows);
void blur_sep_set_slow_counter(unsigned long long *d_counter);
int launch_sobel(cudaStream_t s, const uint8_t *src, uint8_t *dst, int W, int H, int n_frames, int fmt,
                 int src_row0, int src_rows, int out_row0, int out_rows);

// rip_yuv.cu -- camera frames decoded to an interleaved colour image or to the reference's gray: NV12_COLOR and I420 (W and
// H even), YUYV and UYVY (W even), and the Bayer patterns at 8, 10, 12, 14 and 16 bits (W and H at least 3) and packed at 10
// and 12 bits (W a multiple of 4 or 2 and at least 4, H at least 3; kernels in rip_bayer.cu)
inline bool is_packed_bayer(int fmt) { return fmt >= RIP_FMT_BAYER_RGGB10P_MIPI && fmt <= RIP_FMT_BAYER_GBRG12P_GENICAM; }
inline bool is_bayer(int fmt) { return (fmt >= RIP_FMT_BAYER_RGGB8 && fmt <= RIP_FMT_BAYER_GBRG16) || is_packed_bayer(fmt); }
// bits per sample of a Bayer format (8: one byte per pixel; 10 to 16: one little-endian 16-bit word, or packed at 10 and 12),
// 0 for any other format
inline int bayer_bits(int fmt)
{
    if (fmt >= RIP_FMT_BAYER_RGGB8 && fmt <= RIP_FMT_BAYER_GBRG8) return 8;
    if (fmt >= RIP_FMT_BAYER_RGGB10 && fmt <= RIP_FMT_BAYER_GBRG16) return 10 + 2 * ((fmt - RIP_FMT_BAYER_RGGB10) >> 2);
    if (fmt >= RIP_FMT_BAYER_RGGB10P_MIPI && fmt <= RIP_FMT_BAYER_GBRG12P_MIPI) return 10 + 2 * ((fmt - RIP_FMT_BAYER_RGGB10P_MIPI) >> 2);
    if (fmt >= RIP_FMT_BAYER_RGGB10P_GENICAM && fmt <= RIP_FMT_BAYER_GBRG12P_GENICAM)
        return 10 + 2 * ((fmt - RIP_FMT_BAYER_RGGB10P_GENICAM) >> 2);
    return 0;
}
// how a Bayer format stores its samples: whole bytes or 16-bit words, MIPI CSI-2 RAW10 / RAW12, or a GenICam bit stream
enum BayerPacking { BAYER_UNPACKED, BAYER_MIPI, BAYER_GENICAM };
inline int bayer_packing(int fmt)
{
    if (fmt >= RIP_FMT_BAYER_RGGB10P_MIPI && fmt <= RIP_FMT_BAYER_GBRG12P_MIPI) return BAYER_MIPI;
    if (fmt >= RIP_FMT_BAYER_RGGB10P_GENICAM && fmt <= RIP_FMT_BAYER_GBRG12P_GENICAM) return BAYER_GENICAM;
    return BAYER_UNPACKED;
}
inline bool decodes_to_color(int fmt)
{
    return fmt == RIP_FMT_NV12_COLOR || fmt == RIP_FMT_YUYV || fmt == RIP_FMT_UYVY || fmt == RIP_FMT_I420 || is_bayer(fmt);
}
enum YuvOut { YUV_TO_RGB, YUV_TO_BGR, YUV_TO_RGBA, YUV_TO_BGRA, YUV_TO_GRAY, YUV_TO_GRAY_RGBA };
const char *yuv_format_name(int fmt);   // "NV12_COLOR", "YUYV", "UYVY", "I420", "BAYER_RGGB8", ..., "BAYER_GBRG12P_GENICAM"
int check_yuv_shape(int fmt, int W, int H);   // the format's shape rules and the kernels' 32-bit index limit
int launch_yuv(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames, int in_format, YuvOut to);
// rip_bayer.cu -- the demosaic kernels behind launch_yuv; the shape is already checked
int launch_bayer(cudaStream_t s, const uint8_t *in, uint8_t *out, int W, int H, int n_frames, int in_format, YuvOut to);

// rip_fused.cu -- single-kernel gray -> 5x5 Gaussian -> Sobel (and gray -> Sobel)
bool fused_supported(int W, int H, int fmt, int ksize /* 5, or 0 = no blur stage */, const uint8_t *d_in, const uint8_t *d_out);
bool fused_plan_weights(const float *w25, float g[3], float *thr);
void fused_set_slow_counter(unsigned long long *d_counter);
int fused_selftest(int device, unsigned long long *checked, unsigned long long *mismatches);
int launch_fused(cudaStream_t s, const uint8_t *d_in, uint8_t *d_out, int W, int H, int n_frames, int fmt,
                 bool with_blur, const float *weights25, int in_row0, int in_rows, int out_row0, int out_rows,
                 int device);

// rip_fused_tile.cu -- the same pipeline in one kernel for any shape, any odd K <= RIP_MAX_KSIZE, any weights (reference order throughout)
int launch_fused_tile(cudaStream_t s, const uint8_t *d_in, uint8_t *d_out, int W, int H, int n_frames, int fmt, int ksize,
                      const Weights &wts, int in_row0, int in_rows, int out_row0, int out_rows);

}  // namespace rip
