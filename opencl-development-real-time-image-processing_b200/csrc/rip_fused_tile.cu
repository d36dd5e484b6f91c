// rip_fused_tile.cu -- gray -> KxK Gaussian -> 3x3 Sobel in ONE kernel for the shapes the streaming kernel
// (rip_fused_x3.cuh) does not take: any width and height (the reference's own test images are 75, 427, 683 and
// 1023 pixels wide), unaligned buffers, any odd K <= 31 (the reference's default is 17x17, sigma 6:
// include/ProgramHandler.hpp:9), weights that are not a separable kernel.  One HBM round trip like the streaming
// kernel -- round 1 ran these shapes as three kernels through a workspace (gray, blur, Sobel: three round trips).
//
// A block of 256 threads produces a 32 x 16 output tile.  Everything is the reference's own arithmetic, in its
// own order, so there is no fast path and nothing to fix up:
//   1. gray (Comparator.cpp:41) of the tile plus a halo of K/2 + 1 pixels, coordinates clamped to the image
//      (GaussianBlur.cpp:240-241), as bytes in shared memory;
//   2. the blurred tile plus a halo of 1 pixel: float accumulator from 0.0f, taps ky-major / kx-minor, one rounded
//      product and one rounded add per tap (GaussianBlur.cpp:236-258), clamped and truncated to u8.  Halo entries
//      outside the image hold the blurred value of the BORDER_REFLECT_101 coordinate, which is what cv::filter2D
//      reads there (EdgeDetection.cpp:231-233);
//   3. Sobel on the blurred bytes: integer sums, correctly rounded sqrt, round-half-even, saturate
//      (EdgeDetection.cpp:234-240).
#include "rip_common.cuh"
#include "rip_internal.h"

namespace rip {

namespace {

constexpr int FT_TW = 32, FT_TH = 16, FT_THREADS = 256;
constexpr int FT_MAX_HALF = RIP_MAX_KSIZE / 2;
constexpr int FT_GW = FT_TW + 2 + 2 * FT_MAX_HALF, FT_GH = FT_TH + 2 + 2 * FT_MAX_HALF;   // largest gray tile
constexpr int FT_BW = FT_TW + 2, FT_BH = FT_TH + 2;                                        // blurred tile

struct TileParams {
    const uint8_t *src;
    uint8_t *dst;
    int W, H;
    int in_row0, in_rows, out_row0, out_rows;
    size_t in_frame_bytes;
    int ksize;
};

template <int CN, bool BGR>
__global__ void __launch_bounds__(FT_THREADS)
fused_tile_kernel(const TileParams p, const __grid_constant__ Weights wts)
{
    __shared__ uint8_t gray[FT_GH * FT_GW];
    __shared__ uint8_t blur[FT_BH * FT_BW];
    const int W = p.W, H = p.H, half = p.ksize >> 1;
    const int gw = FT_TW + 2 + 2 * half, gh = FT_TH + 2 + 2 * half;
    const int x0 = blockIdx.x * FT_TW, y0 = p.out_row0 + blockIdx.y * FT_TH;
    const int gx0 = x0 - 1 - half, gy0 = y0 - 1 - half;   // image coordinates of gray tile element (0, 0)
    const uint8_t *fsrc = p.src + (size_t)blockIdx.z * p.in_frame_bytes;
    uint8_t *fdst = p.dst + (size_t)blockIdx.z * p.out_rows * W;

    // 1. gray tile (clamp-to-edge coordinates; rows the input band does not hold are never consumed)
    for (int i = threadIdx.x; i < gw * gh; i += FT_THREADS) {
        const int ty = i / gw, tx = i - ty * gw;
        const int cy = clampi(gy0 + ty, 0, H - 1) - p.in_row0, cx = clampi(gx0 + tx, 0, W - 1);
        uint32_t v = 0;
        if (cy >= 0 && cy < p.in_rows) {
            const uint8_t *q = fsrc + ((size_t)cy * W + cx) * CN;
            if (CN == 1) v = q[0];
            else v = BGR ? gray_exact(q[2], q[1], q[0]) : gray_exact(q[0], q[1], q[2]);
        }
        gray[ty * gw + tx] = (uint8_t)v;
    }
    __syncthreads();

    // 2. blurred tile with its 1-pixel BORDER_REFLECT_101 halo
    const int y_end = min(p.out_row0 + p.out_rows, H);
    for (int i = threadIdx.x; i < FT_BW * FT_BH; i += FT_THREADS) {
        const int by = i / FT_BW, bx = i - by * FT_BW;
        const int ry = reflect101(min(y0 - 1 + by, H), H), rx = reflect101(min(x0 - 1 + bx, W), W);
        uint32_t o = 0;
        if (y0 - 1 + by <= y_end && x0 - 1 + bx <= W) {   // (entries further out feed no stored output)
            float acc = 0.0f;
            for (int ky = 0; ky < p.ksize; ky++) {
                const int ty = clampi(ry + ky - half, 0, H - 1) - gy0;
                const uint8_t *row = gray + ty * gw - gx0;
                for (int kx = 0; kx < p.ksize; kx++) {
                    const int cx = clampi(rx + kx - half, 0, W - 1);
                    acc = __fadd_rn(acc, __fmul_rn((float)row[cx], wts.w[ky * p.ksize + kx]));
                }
            }
            o = (uint32_t)__float2int_rz(fminf(fmaxf(acc, 0.0f), 255.0f));
        }
        blur[i] = (uint8_t)o;
    }
    __syncthreads();

    // 3. Sobel: two horizontally adjacent outputs per thread
    const int tx2 = (threadIdx.x & 15) * 2, ty = threadIdx.x >> 4;
    const int y = y0 + ty;
    if (y >= y_end) return;
    const uint8_t *r0 = blur + ty * FT_BW + tx2, *r1 = r0 + FT_BW, *r2 = r1 + FT_BW;
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int x = x0 + tx2 + i;
        if (x >= W) break;
        const int a = r0[i], b = r0[i + 1], c = r0[i + 2];
        const int d = r1[i], f = r1[i + 2];
        const int g = r2[i], h = r2[i + 1], k = r2[i + 2];
        const int gx = (c - a) + 2 * (f - d) + (k - g);
        const int gy = (g - a) + 2 * (h - b) + (k - c);
        fdst[(size_t)(y - p.out_row0) * W + x] = (uint8_t)sobel_mag(gx, gy);
    }
}

}  // namespace

int launch_fused_tile(cudaStream_t s, const uint8_t *d_in, uint8_t *d_out, int W, int H, int n_frames, int fmt, int ksize,
                      const Weights &wts, int in_row0, int in_rows, int out_row0, int out_rows)
{
    if (ksize < 1 || ksize > RIP_MAX_KSIZE || !(ksize & 1)) return fail(RIP_EINVAL, "rip_fused: kernel size must be odd and in [1,%d]", RIP_MAX_KSIZE);
    TileParams p;
    p.src = d_in; p.dst = d_out; p.W = W; p.H = H;
    p.in_row0 = in_row0; p.in_rows = in_rows; p.out_row0 = out_row0; p.out_rows = out_rows;
    p.ksize = ksize;
    const Format &f = *format_of(fmt);   // (rip_fused checked the format)
    // whole NV12 frames carry their chroma plane behind the luma plane; row bands are passed as plain luma rows
    p.in_frame_bytes = (in_row0 == 0 && in_rows == H) ? frame_bytes(f, W, H) : (size_t)in_rows * W * f.channels;
    // frames ride in gridDim.z (<= 65535): batches of tiny frames go out in slabs
    for (int f0 = 0; f0 < n_frames; f0 += kMaxGridZ) {
        const dim3 grid((W + FT_TW - 1) / FT_TW, (out_rows + FT_TH - 1) / FT_TH, min(n_frames - f0, kMaxGridZ));
        TileParams q = p;
        q.src = d_in + (size_t)f0 * p.in_frame_bytes;
        q.dst = d_out + (size_t)f0 * out_rows * W;
        switch (fmt) {
        case RIP_FMT_GRAY8: case RIP_FMT_NV12: fused_tile_kernel<1, false><<<grid, FT_THREADS, 0, s>>>(q, wts); break;
        case RIP_FMT_RGB8:  fused_tile_kernel<3, false><<<grid, FT_THREADS, 0, s>>>(q, wts); break;
        case RIP_FMT_BGR8:  fused_tile_kernel<3, true><<<grid, FT_THREADS, 0, s>>>(q, wts); break;
        case RIP_FMT_RGBA8: fused_tile_kernel<4, false><<<grid, FT_THREADS, 0, s>>>(q, wts); break;
        case RIP_FMT_BGRA8: fused_tile_kernel<4, true><<<grid, FT_THREADS, 0, s>>>(q, wts); break;
        default: return fail(RIP_EINVAL, "rip_fused: unsupported input format %d", fmt);
        }
        RIP_LAUNCH_CHECK();
    }
    return RIP_OK;
}

}  // namespace rip
