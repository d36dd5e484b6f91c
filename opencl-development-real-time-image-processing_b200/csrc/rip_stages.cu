// rip_stages.cu -- the three stand-alone stages (gray, KxK Gaussian, 3x3 Sobel) as sm_100a kernels.
//
// These replace kernel/grayscale_base.cl, gaussian_base.cl and edge_base.cl of the reference, but
// compute what the reference's CPU paths compute (the parity oracle), not what its OpenCL kernels
// compute: see rip_common.cuh for the arithmetic.  The generic-K blur here is the exact
// reference-order kernel (the "truth" path); the single-pass fused pipeline lives in rip_fused.cu.
#include <type_traits>

#include "rip_common.cuh"
#include "rip_internal.h"

namespace rip {

// ---------------------------------------------------------------------------------------------
// gray: pointwise, 4 pixels per thread, 128-bit loads (RGBA) / 3 x 32-bit loads (RGB),
// 32-bit (u8 out) or 128-bit ((g,g,g,255) out) stores.  5 or 8 algorithmic bytes per pixel.
// ---------------------------------------------------------------------------------------------
template <int CN, bool BGR, bool OUT_RGBA>
__global__ void __launch_bounds__(256)
gray_kernel(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, long long npx)
{
    const long long nquad = npx >> 2;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nquad; q += stride) {
        uint32_t c0[4], c1[4], c2[4];  // channel 0/1/2 of the four pixels
        if (CN == 4) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(in) + q);
            const uint32_t p[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int i = 0; i < 4; i++) {
                c0[i] = p[i] & 0xffu;
                c1[i] = (p[i] >> 8) & 0xffu;
                c2[i] = (p[i] >> 16) & 0xffu;
            }
        } else {
            const uint32_t *p = reinterpret_cast<const uint32_t *>(in) + q * 3;
            const uint32_t w0 = __ldg(p), w1 = __ldg(p + 1), w2 = __ldg(p + 2);
            c0[0] = w0 & 0xffu;         c1[0] = (w0 >> 8) & 0xffu;  c2[0] = (w0 >> 16) & 0xffu;
            c0[1] = w0 >> 24;           c1[1] = w1 & 0xffu;         c2[1] = (w1 >> 8) & 0xffu;
            c0[2] = (w1 >> 16) & 0xffu; c1[2] = w1 >> 24;           c2[2] = w2 & 0xffu;
            c0[3] = (w2 >> 8) & 0xffu;  c1[3] = (w2 >> 16) & 0xffu; c2[3] = w2 >> 24;
        }
        uint32_t y[4];
#pragma unroll
        for (int i = 0; i < 4; i++) y[i] = BGR ? gray_exact(c2[i], c1[i], c0[i]) : gray_exact(c0[i], c1[i], c2[i]);
        if (OUT_RGBA) {
            uint4 o;
            o.x = y[0] * 0x010101u | 0xff000000u;
            o.y = y[1] * 0x010101u | 0xff000000u;
            o.z = y[2] * 0x010101u | 0xff000000u;
            o.w = y[3] * 0x010101u | 0xff000000u;
            reinterpret_cast<uint4 *>(out)[q] = o;
        } else {
            reinterpret_cast<uint32_t *>(out)[q] = y[0] | (y[1] << 8) | (y[2] << 16) | (y[3] << 24);
        }
    }
    // tail (npx % 4 pixels), one thread each
    const long long i = (nquad << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < npx) {
        const uint8_t *p = in + i * CN;
        const uint32_t y = BGR ? gray_exact(p[2], p[1], p[0]) : gray_exact(p[0], p[1], p[2]);
        if (OUT_RGBA) {
            reinterpret_cast<uint32_t *>(out)[i] = y * 0x010101u | 0xff000000u;
        } else {
            out[i] = (uint8_t)y;
        }
    }
}

// byte-granular variant for buffers whose base is not 16-byte aligned
template <int CN, bool BGR, bool OUT_RGBA>
__global__ void __launch_bounds__(256)
gray_kernel_unaligned(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, long long npx)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += stride) {
        const uint8_t *p = in + i * CN;
        const uint32_t y = BGR ? gray_exact(p[2], p[1], p[0]) : gray_exact(p[0], p[1], p[2]);
        if (OUT_RGBA) {
            out[4 * i] = out[4 * i + 1] = out[4 * i + 2] = (uint8_t)y;
            out[4 * i + 3] = 255;
        } else {
            out[i] = (uint8_t)y;
        }
    }
}

template <int CN, bool BGR>
static int launch_gray_t(cudaStream_t s, const uint8_t *in, uint8_t *out, long long npx, int out_mode, int device)
{
    const bool aligned = ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0;
    const long long work = aligned ? ((npx + 3) >> 2) : npx;
    long long blocks = (work + 255) / 256;
    const long long cap = (long long)sm_count(device) * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    const dim3 grid((unsigned)blocks), block(256);
    if (aligned) {
        if (out_mode == RIP_GRAY_OUT_RGBA) gray_kernel<CN, BGR, true><<<grid, block, 0, s>>>(in, out, npx);
        else gray_kernel<CN, BGR, false><<<grid, block, 0, s>>>(in, out, npx);
    } else {
        if (out_mode == RIP_GRAY_OUT_RGBA) gray_kernel_unaligned<CN, BGR, true><<<grid, block, 0, s>>>(in, out, npx);
        else gray_kernel_unaligned<CN, BGR, false><<<grid, block, 0, s>>>(in, out, npx);
    }
    RIP_LAUNCH_CHECK();
    return RIP_OK;
}

int launch_gray(cudaStream_t s, const uint8_t *in, uint8_t *out, long long npx, int fmt, int out_mode, int device)
{
    switch (fmt) {
    case RIP_FMT_RGB8:  return launch_gray_t<3, false>(s, in, out, npx, out_mode, device);
    case RIP_FMT_BGR8:  return launch_gray_t<3, true>(s, in, out, npx, out_mode, device);
    case RIP_FMT_RGBA8: return launch_gray_t<4, false>(s, in, out, npx, out_mode, device);
    case RIP_FMT_BGRA8: return launch_gray_t<4, true>(s, in, out, npx, out_mode, device);
    default: return fail(RIP_EINVAL, "rip_gray: unsupported input format %d", fmt);
    }
}

// ---------------------------------------------------------------------------------------------
// KxK Gaussian, exact reference order (GaussianBlur.cpp:236-258): per channel one fp32 accumulator
// from 0.0f, taps ky-major / kx-minor, product rounded, then sum rounded (no FMA), clamp-to-edge
// coordinates, clamp to [0,255], truncate.  Tile with halo staged in shared memory.
// ---------------------------------------------------------------------------------------------
constexpr int BLUR_TW = 32, BLUR_TH = 8;

template <int CN>
__global__ void __launch_bounds__(BLUR_TW *BLUR_TH)
blur_exact_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int W, int H, int src_row0,
                  int src_rows, int out_row0, int out_rows, int ksize, const __grid_constant__ Weights wts)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    using px_t = typename std::conditional<CN == 4, uint32_t, uint8_t>::type;
    px_t *tile = reinterpret_cast<px_t *>(smem_raw);

    const int half = ksize >> 1;
    const int tw = BLUR_TW + 2 * half, th = BLUR_TH + 2 * half;
    const int x0 = blockIdx.x * BLUR_TW, y0 = out_row0 + blockIdx.y * BLUR_TH;
    const px_t *fsrc = reinterpret_cast<const px_t *>(src) + (size_t)blockIdx.z * src_rows * W;
    px_t *fdst = reinterpret_cast<px_t *>(dst) + (size_t)blockIdx.z * out_rows * W;
    const int tid = threadIdx.y * BLUR_TW + threadIdx.x;

    // rows past the last output row of this band (+halo) are never consumed and may lie outside src
    const int y_last = min(out_row0 + out_rows, H) - 1 + half;
    for (int i = tid; i < tw * th; i += BLUR_TW * BLUR_TH) {
        const int ty = i / tw, tx = i - ty * tw;
        px_t v = 0;
        if (y0 - half + ty <= y_last) {
            const int gy = clampi(y0 - half + ty, 0, H - 1);
            const int gx = clampi(x0 - half + tx, 0, W - 1);
            v = fsrc[(size_t)(gy - src_row0) * W + gx];
        }
        tile[i] = v;
    }
    __syncthreads();

    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= W || y >= out_row0 + out_rows || y >= H) return;

    float acc[CN];
#pragma unroll
    for (int c = 0; c < CN; c++) acc[c] = 0.0f;
    for (int ky = 0; ky < ksize; ky++) {
        const px_t *row = tile + (threadIdx.y + ky) * tw + threadIdx.x;
        for (int kx = 0; kx < ksize; kx++) {
            const float w = wts.w[ky * ksize + kx];
            const uint32_t p = row[kx];
#pragma unroll
            for (int c = 0; c < CN; c++) {
                const float v = (float)((p >> (8 * c)) & 0xffu);
                acc[c] = __fadd_rn(acc[c], __fmul_rn(v, w));
            }
        }
    }
    uint32_t o = 0;
#pragma unroll
    for (int c = 0; c < CN; c++) {
        const float v = fminf(fmaxf(acc[c], 0.0f), 255.0f);
        o |= (uint32_t)__float2int_rz(v) << (8 * c);
    }
    fdst[(size_t)(y - out_row0) * W + x] = (px_t)o;
}

int launch_blur_exact(cudaStream_t s, const uint8_t *src, uint8_t *dst, int W, int H, int n_frames, int cn,
                      int ksize, const Weights &wts, int src_row0, int src_rows, int out_row0, int out_rows)
{
    if (cn != 1 && cn != 4) return fail(RIP_EINVAL, "rip_gauss: channels must be 1 or 4 (got %d)", cn);
    if (cn == 4 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 3u))
        return fail(RIP_EINVAL, "rip_gauss: RGBA buffers must be 4-byte aligned");
    const int half = ksize >> 1;
    const dim3 block(BLUR_TW, BLUR_TH);
    const size_t smem = (size_t)(BLUR_TW + 2 * half) * (BLUR_TH + 2 * half) * cn;
    // frames ride in gridDim.z (<= 65535): batches of tiny frames go out in slabs
    for (int f0 = 0; f0 < n_frames; f0 += kMaxGridZ) {
        const int nf = min(n_frames - f0, kMaxGridZ);
        const dim3 grid((W + BLUR_TW - 1) / BLUR_TW, (out_rows + BLUR_TH - 1) / BLUR_TH, nf);
        const uint8_t *fs = src + (size_t)f0 * src_rows * W * cn;
        uint8_t *fd = dst + (size_t)f0 * out_rows * W * cn;
        if (cn == 4)
            blur_exact_kernel<4><<<grid, block, smem, s>>>(fs, fd, W, H, src_row0, src_rows, out_row0, out_rows, ksize, wts);
        else
            blur_exact_kernel<1><<<grid, block, smem, s>>>(fs, fd, W, H, src_row0, src_rows, out_row0, out_rows, ksize, wts);
        RIP_LAUNCH_CHECK();
    }
    return RIP_OK;
}

int launch_blur(cudaStream_t s, const uint8_t *src, uint8_t *dst, int W, int H, int n_frames, int cn,
                int ksize, const Weights &wts, int src_row0, int src_rows, int out_row0, int out_rows)
{
    const int rc = launch_blur_sep(s, src, dst, W, H, n_frames, cn, ksize, wts, src_row0, src_rows, out_row0, out_rows);
    if (rc != RIP_EUNSUPPORTED) return rc;
    return launch_blur_exact(s, src, dst, W, H, n_frames, cn, ksize, wts, src_row0, src_rows, out_row0, out_rows);
}

// ---------------------------------------------------------------------------------------------
// 3x3 Sobel magnitude (OpenCV semantics).  A 64x16 output tile per block; the gray tile with its
// 1-pixel BORDER_REFLECT_101 halo is built in shared memory (converted from colour on the fly when
// the input is not already gray); each thread then produces 4 horizontally adjacent pixels.
// ---------------------------------------------------------------------------------------------
constexpr int SOB_TW = 64, SOB_TH = 16, SOB_SW = SOB_TW + 2 + 2 /* pad to a multiple of 4 */;

template <int CN, bool BGR>
__global__ void __launch_bounds__(256)
sobel_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int W, int H, int src_row0, int src_rows,
             int out_row0, int out_rows, size_t in_frame_bytes)
{
    __shared__ uint8_t tile[(SOB_TH + 2) * SOB_SW];
    const int x0 = blockIdx.x * SOB_TW, y0 = out_row0 + blockIdx.y * SOB_TH;
    const uint8_t *fsrc = src + (size_t)blockIdx.z * in_frame_bytes;
    uint8_t *fdst = dst + (size_t)blockIdx.z * out_rows * W;
    const int y_end = min(out_row0 + out_rows, H);

    for (int i = threadIdx.x; i < (SOB_TH + 2) * (SOB_TW + 2); i += 256) {
        const int ty = i / (SOB_TW + 2), tx = i - ty * (SOB_TW + 2);
        const int gy = reflect101(min(y0 - 1 + ty, H), H);
        const int gx = reflect101(min(x0 - 1 + tx, W), W);
        uint32_t v = 0;
        if (y0 - 1 + ty <= y_end) {  // rows beyond the band are never consumed
            const uint8_t *p = fsrc + ((size_t)(gy - src_row0) * W + gx) * CN;
            if (CN == 1) v = p[0];
            else v = BGR ? gray_exact(p[2], p[1], p[0]) : gray_exact(p[0], p[1], p[2]);
        }
        tile[ty * SOB_SW + tx] = (uint8_t)v;
    }
    __syncthreads();

    const int tx4 = (threadIdx.x & 15) * 4, ty = threadIdx.x >> 4;
    const int y = y0 + ty;
    if (y >= y_end) return;
    const uint8_t *r0 = tile + ty * SOB_SW + tx4, *r1 = r0 + SOB_SW, *r2 = r1 + SOB_SW;
    uint32_t o[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int a = r0[i], b = r0[i + 1], c = r0[i + 2];
        const int d = r1[i], f = r1[i + 2];
        const int g = r2[i], h = r2[i + 1], k = r2[i + 2];
        const int gx = (c - a) + 2 * (f - d) + (k - g);
        const int gy = (g - a) + 2 * (h - b) + (k - c);
        o[i] = sobel_mag(gx, gy);
    }
    const int x = x0 + tx4;
    uint8_t *orow = fdst + (size_t)(y - out_row0) * W;
    if (x + 3 < W && ((reinterpret_cast<uintptr_t>(orow + x) & 3u) == 0)) {
        *reinterpret_cast<uint32_t *>(orow + x) = o[0] | (o[1] << 8) | (o[2] << 16) | (o[3] << 24);
    } else {
#pragma unroll
        for (int i = 0; i < 4; i++)
            if (x + i < W) orow[x + i] = (uint8_t)o[i];
    }
}

int launch_sobel(cudaStream_t s, const uint8_t *src, uint8_t *dst, int W, int H, int n_frames, int fmt,
                 int src_row0, int src_rows, int out_row0, int out_rows)
{
    const dim3 block(256);
    const Format &f = *format_of(fmt);   // (rip_sobel checked the format)
    // whole NV12 frames carry their chroma plane behind the luma plane; row bands are passed as plain luma rows
    const size_t in_frame_bytes = (src_row0 == 0 && src_rows == H) ? frame_bytes(f, W, H) : (size_t)src_rows * W * f.channels;
    // frames ride in gridDim.z (<= 65535): batches of tiny frames go out in slabs
    for (int f0 = 0; f0 < n_frames; f0 += kMaxGridZ) {
        const dim3 grid((W + SOB_TW - 1) / SOB_TW, (out_rows + SOB_TH - 1) / SOB_TH, min(n_frames - f0, kMaxGridZ));
        const uint8_t *fs = src + (size_t)f0 * in_frame_bytes;
        uint8_t *fd = dst + (size_t)f0 * out_rows * W;
#define RIP_SOBEL_CASE(F, CN, BGR) \
    case F: sobel_kernel<CN, BGR><<<grid, block, 0, s>>>(fs, fd, W, H, src_row0, src_rows, out_row0, out_rows, in_frame_bytes); break;
        switch (fmt) {
            RIP_SOBEL_CASE(RIP_FMT_GRAY8, 1, false)
            RIP_SOBEL_CASE(RIP_FMT_NV12, 1, false)
            RIP_SOBEL_CASE(RIP_FMT_RGB8, 3, false)
            RIP_SOBEL_CASE(RIP_FMT_BGR8, 3, true)
            RIP_SOBEL_CASE(RIP_FMT_RGBA8, 4, false)
            RIP_SOBEL_CASE(RIP_FMT_BGRA8, 4, true)
        default: return fail(RIP_EINVAL, "rip_sobel: unsupported input format %d", fmt);
        }
#undef RIP_SOBEL_CASE
        RIP_LAUNCH_CHECK();
    }
    return RIP_OK;
}

}  // namespace rip
