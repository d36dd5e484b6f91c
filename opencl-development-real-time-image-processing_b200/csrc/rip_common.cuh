// rip_common.cuh -- shared device helpers and host-side error plumbing for librip_cuda.so.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "rip_cuda.h"

#define RIP_MAX_TAPS (RIP_MAX_KSIZE * RIP_MAX_KSIZE)

namespace rip {

// ---- host side -------------------------------------------------------------------------------
int fail(int code, const char *fmt, ...);                       // records thread-local message
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);
void count_launch(uint64_t n = 1);

#define RIP_CUDA(call)                                                        \
    do {                                                                      \
        cudaError_t _e = (call);                                              \
        if (_e != cudaSuccess) return rip::cuda_fail(_e, #call, __FILE__, __LINE__); \
    } while (0)

#define RIP_LAUNCH_CHECK()                                                    \
    do {                                                                      \
        cudaError_t _e = cudaGetLastError();                                  \
        if (_e != cudaSuccess) return rip::cuda_fail(_e, "kernel launch", __FILE__, __LINE__); \
        rip::count_launch();                                                  \
    } while (0)

// RAII device switch: every entry point names its device explicitly.
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; }
        if (prev != dev) ok = (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

int sm_count(int device);
constexpr int kMaxGridZ = 65535;   // frames per launch of the kernels that index frames with blockIdx.z

// Debug / experiment switches.  Read from the environment ONCE (first use), then only changed through
// rip_debug_set_option(): no getenv() on any launch path.
struct Options {
    int fused_seg = 0;       // RIP_FUSED_SEG:     rows per segment of the fused kernel (0 = automatic)
    int fused_npx = 0;       // RIP_FUSED_NPX:     4 = force the 4-pixel-per-lane kernel (0 / 8 = automatic)
    int fused_generic = 0;   // RIP_FUSED_GENERIC: rip_fused always runs the any-shape tile kernel (rip_fused_tile.cu)
    int blur_exact = 0;      // RIP_BLUR_EXACT:    always run the reference-order blur kernel
    int blur_tiled = 0;      // RIP_BLUR_TILED:    never run the streaming blur kernels
    int blur_stream = 0;     // RIP_BLUR_STREAM:   run the streaming blur kernels on small inputs too
};
const Options &options();

// KxK weights passed by value: lives in the kernel-parameter constant bank, so every tap is a
// uniform constant-cache read and concurrent streams can use different kernels safely.
struct Weights {
    float w[RIP_MAX_TAPS];
};

// ---- device side -----------------------------------------------------------------------------

// Reference gray (Comparator.cpp:41): (uchar)(0.299*r + 0.587*g + 0.114*b) evaluated in double,
// left to right, truncated.  With t = 299r + 587g + 114b the real value is t/1000; whenever
// t % 1000 != 0 it sits >= 1e-3 away from an integer while the double evaluation is off by
// < 1e-12, so floor(t/1000) is exact.  Only on exact multiples of 1000 (0.1 % of triples, but
// every r=g=b grey) does the rounding of the three double products decide between q and q-1;
// those pixels replay the double sequence with explicitly unfused operations.
__device__ __forceinline__ uint32_t gray_exact(uint32_t r, uint32_t g, uint32_t b)
{
    const uint32_t t = 299u * r + 587u * g + 114u * b;
    uint32_t q = t / 1000u;
    if (t - q * 1000u == 0u) {
        const double s = __dadd_rn(__dadd_rn(__dmul_rn(0.299, (double)r), __dmul_rn(0.587, (double)g)),
                                   __dmul_rn(0.114, (double)b));
        q = (uint32_t)__double2int_rz(s);
    }
    return q;
}

__device__ __forceinline__ int reflect101(int i, int n)
{
    // cv::BORDER_REFLECT_101 for |overshoot| <= 1 (3x3 kernels); a length-1 axis maps to 0.
    if (n == 1) return 0;
    if (i < 0) return -i;
    if (i >= n) return 2 * (n - 1) - i;
    return i;
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return min(max(v, lo), hi); }

// OpenCV Sobel magnitude (EdgeDetection.cpp:231-240): gx, gy are exact small integers,
// gx*gx+gy*gy < 2^24 is exact in float, sqrt is correctly rounded, convertTo rounds half to even
// and saturates.
__device__ __forceinline__ uint32_t sobel_mag(int gx, int gy)
{
    const float m = __fsqrt_rn((float)(gx * gx + gy * gy));
    return (uint32_t)min(__float2int_rn(m), 255);
}

}  // namespace rip
