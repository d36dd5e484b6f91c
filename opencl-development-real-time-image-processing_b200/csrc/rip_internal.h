// rip_internal.h -- launchers shared between the translation units of librip_cuda.so (not exported).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "rip_common.cuh"
#include "rip_formats.h"

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

// rip_yuv.cu -- camera frames (the formats decodes_to_color() names, rip_formats.h) decoded to an interleaved colour image or
// to the reference's gray (Bayer kernels in rip_bayer.cu)
enum YuvOut { YUV_TO_RGB, YUV_TO_BGR, YUV_TO_RGBA, YUV_TO_BGRA, YUV_TO_GRAY, YUV_TO_GRAY_RGBA };
int check_yuv_shape(int fmt, int W, int H);   // the format's shape rule (its row) and the kernels' 32-bit index limit
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
