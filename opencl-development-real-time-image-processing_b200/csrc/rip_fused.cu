// rip_fused.cu -- gray -> 5x5 Gaussian -> 3x3 Sobel in ONE kernel (one HBM round trip per frame), and the
// same kernel without the blur stage (gray -> Sobel, BASELINE config 3): host side (weight planning, grid
// shaping, launch) and the on-device self-test.  The kernel itself is rip_fused_x3.cuh.
//
// Design (sm_100a, an FMA-pipe/issue-bound integer+fp32 stencil; no tensor cores by design):
//   * every WARP is independent.  A lane owns NPX = 8 (or 4) horizontally adjacent pixels; a warp covers
//     32*NPX pixels of which the middle 30*NPX (lanes 1..30) are outputs and the outer lanes are halo.
//     The warp slides DOWN a segment of rows, so the vertical halo costs 6 warm-up rows per segment and
//     the horizontal halo 2/32 of the lanes.  One block-level barrier at start-up, none afterwards.
//   * per image row a lane fetches its 3*NPX (RGB) or 4*NPX (RGBA) bytes into shared memory with cp.async
//     three (with the blur stage) or six rows ahead, converts them to the reference's exact gray, and keeps
//     the vertical blur accumulators and two rows of Sobel input in registers.
//   * the horizontal neighbours (2 per side for the blur, 1 per side for Sobel) come from the adjacent
//     lanes with warp shuffles.
//   * exactness: the blurred value must equal the reference's sequential, unfused, 25-tap fp32 sum
//     truncated to u8 (GaussianBlur.cpp:236-258).  The fast path evaluates a separable fp32 sum S~; a
//     pixel whose S~ is closer to an integer than the proven bound on |S~ - S_ref| (plan_weights_band
//     below) is recomputed with the exact 25-tap sequence.  So the u8 blurred image, and with it the
//     Sobel output, is bit-exact, at separable cost on all but ~0.07 % of the pixels.
//   * Sobel: exact small-integer sums in fp32, magnitude via sqrt.approx (its error is 8x below the
//     distance of any integer's root to a rounding boundary for results < 255.5), round-half-even and
//     saturation by a denormal multiply + I2IP, one 64-bit store per lane per row.
// Earlier kernels of this round (4 px per lane scalar fp32 with direct loads; the same with TMA-staged
// tiles, tools/tma_probe.cu) are described with their measurements in profiles/ and DESIGN.md.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "rip_common.cuh"
#include "rip_internal.h"

namespace rip {

namespace {

constexpr int kWarpsPerBlock = 4;
// x2 kernel (rip_fused_x3.cuh): resident blocks per SM for 8 / 4 pixels per lane
constexpr int kMinBlocks8 = 4;
constexpr int kMinBlocks8NoBlur = 6;   // colour -> gray -> Sobel: six blocks (24 warps) per SM since the row buffers left the registers (76 registers; config 3: 121 -> 117 us; five before: 127 -> 123 us; gray input is better off with 4)
constexpr int kMinBlocks4 = 6;
constexpr unsigned FULL = 0xffffffffu;

struct FusedParams {
    const uint8_t *in;
    uint8_t *out;
    int W, H;
    int in_row0, in_rows, out_row0, out_rows;
    size_t in_frame_bytes;   // distance between the frames of the input batch (NV12: the luma plane plus the chroma plane)
    int seg_rows, n_segs, n_bands, n_band_groups;
    float w[25];         // exact 2-D weights for the replay
    unsigned long long *slow_counter;  // optional statistics (NULL in production)
};

// Exact gray (Comparator.cpp:41).  With t = 299r + 587g + 114b the real value is t/1000; off the
// multiples of 1000 the reference's double expression truncates to q = floor(t/1000) (it is >= 1e-3
// away from an integer, the double rounding error is < 1e-12).  ON a multiple of 1000 the rounding of
// the three double products decides between q and q-1: those pixels (0.1 %) evaluate the reference
// expression itself in double on the device (rip_fused_x3.cuh, gray_down_mask).
__device__ __forceinline__ float sqrt_approx(float x)
{
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

#include "rip_fused_x3.cuh"

}  // namespace

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
bool fused_supported(int W, int H, int fmt, int ksize, const uint8_t *d_in, const uint8_t *d_out)
{
    if (ksize != 0 && ksize != 5) return false;
    if (W < 4 || (W & 3) || H < 2) return false;
    const Format *f = format_of(fmt);
    if (!f || decodes_to_color(fmt) || !shape_ok(*f, W, H)) return false;
    const uintptr_t in_align = f->channels == 4 ? 15u : 3u;
    if ((reinterpret_cast<uintptr_t>(d_in) & in_align) || (reinterpret_cast<uintptr_t>(d_out) & 3u)) return false;
    return true;
}

// half an ulp of the fp32 binade that holds x (x > 0): the largest rounding error of a result whose magnitude is <= x
static double hulp(double x) { return x > 0.0 ? std::ldexp(1.0, (int)std::floor(std::log2(x)) - 24) : 0.0; }

// Guard band for the fast path, and the separable taps that minimise it: a rigorous bound on |S~ - S_ref|, every rounding
// bounded by half an ulp of the BINADE its result can reach (round 1 used u * |value|, up to twice as much; the band went
// from 14 to 8 ulps of 2^-15 for the reference's weights, i.e. 40 % fewer guard-band pixels).  With gray values <= 255,
// w_k the 25 weights in the reference's order, W_k = w_0 + .. + w_k, g the separable taps (floats) and G = g0 + 2 g1 + 2 g2:
//   reference (GaussianBlur.cpp:236-258: acc_k = fl(acc_{k-1} + fl(p_k w_k)), acc_0 = fl(p_0 w_0)):
//     |S_ref - S| <= sum_k hulp(255 w_k) + sum_{k>=1} hulp(255 W_k)
//   separable model in exact arithmetic:        |S_sep - S| <= 255 sum_ij |w_ij - g_i g_j|
//   fast path (rip_fused_x3.cuh): the vertical pass rounds three times (five in the accumulate form; the larger bound is
//     used), |V - V_exact| <= E_V; the pair sums e = fl(V + V') once more, <= E_e = hulp(510 G); the horizontal chain
//     fl(g0 V + bias), fl(g1 e1 + .), fl(g2 e2 + .) rounds on the 2^-16 grid of [256, 512): its last rounding is the +1/2
//     ulp in the choice of `a` (launch_fused_x2_n), the two inner ones add 2 * 2^-16:
//     |S~ - S_sep| <= G E_V + (g1 + g2) E_e + 2^-15
// (all scalings by powers of two in the kernel are exact and keep every intermediate a normal float, checked below).
static bool plan_weights_band(const float *w25, float g[3], double *band_out)
{
    double sum = 0.0;
    for (int i = 0; i < 25; i++) {
        if (!(w25[i] >= 0.0f) || !std::isfinite(w25[i])) return false;
        // the kernel feeds gray in as q * 2^-149 and carries the 2^149 in the weights; a product must
        // stay a normal float for its rounding to equal the reference's (rip_fused_x3.cuh)
        if (w25[i] != 0.0f && w25[i] < 8.470329472543003e-22f /* 2^-70 */) return false;
        sum += (double)w25[i];
    }
    if (!(sum > 0.0) || 255.0 * sum >= 255.9) return false;  // floor(S) must stay <= 255
    // symmetric separable fit from the diagonal: g_k = sqrt(w[k][k])
    for (int k = 0; k < 3; k++) g[k] = (float)std::sqrt((double)w25[(2 + k) * 5 + (2 + k)]);
    const double g0 = g[0], g1 = g[1], g2 = g[2], G = g0 + 2 * g1 + 2 * g2;
    double dev = 0.0;
    for (int ky = -2; ky <= 2; ky++)
        for (int kx = -2; kx <= 2; kx++)
            dev += std::fabs((double)w25[(ky + 2) * 5 + (kx + 2)] - (double)g[std::abs(ky)] * (double)g[std::abs(kx)]);
    const double up = 1.0 + 1e-6;   // (bounds that sit just below a power of two are pushed into the next binade: safe side)
    double b_ref = 0.0, cumw = 0.0;
    for (int k = 0; k < 25; k++) {
        cumw += (double)w25[k];
        b_ref += hulp(255.0 * w25[k] * up);
        if (k >= 1) b_ref += hulp(255.0 * cumw + 1e-3);   // (+1e-3: the computed partial sums carry their own errors)
    }
    const double e_v = hulp(255.0 * g2 * up) + hulp(255.0 * (g2 + g1) * up) + hulp(255.0 * (g2 + g1 + g0) * up) +
                       hulp(255.0 * (g2 + 2 * g1 + g0) * up) + hulp(255.0 * G * up);
    const double e_e = hulp(510.0 * G * up);
    const double b_fast = G * e_v + (g1 + g2) * e_e + std::ldexp(1.0, -15);
    const double band = (255.0 * dev + b_ref + b_fast) * 1.01 + 1e-7;
    if (band > 0.05) return false;  // weights are not (close to) a symmetric separable kernel
    *band_out = band;
    return true;
}

bool fused_plan_weights(const float *w25, float g[3], float *thr)
{
    double band;
    if (!plan_weights_band(w25, g, &band)) return false;
    *thr = (float)(0.5 - band);
    return true;
}

static int pick_seg_rows(int out_rows, int n_frames, int n_band_groups, int device, int resident_blocks = 6)
{
    if (const int v = options().fused_seg; v > 0) return v < out_rows ? v : out_rows;
    // enough blocks for >= ~3 waves of (SMs x resident blocks), but segments of >= 32 rows (6 warm-up rows
    // each); never more than 256 rows (tail balance).  Measured: 32 4K frames 94..270 rows 416-430 us (flat),
    // 360 rows 500 us; a single 4K frame 32 rows 38 us, 64 rows 46 us, 128 rows 67 us.
    const long long target_blocks = (long long)sm_count(device) * resident_blocks * 3;
    int seg = 256;
    while (seg > 32 && (long long)n_frames * n_band_groups * ((out_rows + seg - 1) / seg) < target_blocks) seg >>= 1;
    if (seg > out_rows) seg = out_rows;
    return seg;
}

static unsigned long long *g_slow_counter = nullptr;  // set by rip_debug_slow_path_stats

// bit v of flat_dec: the reference's sum over a CONSTANT 5x5 window of gray value v (GaussianBlur.cpp:236-258: float
// accumulator from 0.0f, ky-major / kx-minor, one rounded product and one rounded add per tap) truncates to one
// below the nearest integer.  Evaluated with the reference's own sequence for the weights in use; the kernel's
// flat-region shortcut reads it instead of replaying 25 taps per pixel.
static void plan_flat_table(const float *w25, uint32_t flat_dec[8])
{
    memset(flat_dec, 0, 8 * sizeof(uint32_t));
    for (int v = 0; v < 256; v++) {
        volatile float acc = 0.0f;   // volatile: every product and every add is rounded to float, none is fused
        for (int i = 0; i < 25; i++) {
            volatile float prod = (float)v * w25[i];
            acc = acc + prod;
        }
        const float s = acc;
        if (s < rintf(s)) flat_dec[v >> 5] |= 1u << (v & 31);
    }
}

// ---- x2 kernel (the default) --------------------------------------------------------------------
template <int NPX, int CN, bool BGR>
static void launch_x2_t(bool blur, dim3 grid, cudaStream_t s, const X2Params &xp)
{
    if (blur && xp.f.slow_counter) fused_x2_kernel<NPX, CN, BGR, true, true><<<grid, kWarpsPerBlock * 32, 0, s>>>(xp);   // (statistics build)
    else if (blur) fused_x2_kernel<NPX, CN, BGR, true><<<grid, kWarpsPerBlock * 32, 0, s>>>(xp);
    else fused_x2_kernel<NPX, CN, BGR, false><<<grid, kWarpsPerBlock * 32, 0, s>>>(xp);
}

template <int NPX>
static int launch_fused_x2_n(cudaStream_t s, FusedParams p, int n_frames, int fmt, bool with_blur, double band, const float g[3], int device)
{
    constexpr int kBand = 30 * NPX;
    X2Params xp;
    memset(&xp, 0, sizeof(xp));
    p.n_bands = (p.W + kBand - 1) / kBand;
    p.n_band_groups = (p.n_bands + kWarpsPerBlock - 1) / kWarpsPerBlock;
    p.seg_rows = pick_seg_rows(p.out_rows, n_frames, p.n_band_groups, device, NPX == 8 ? kMinBlocks8 : kMinBlocks4);
    p.n_segs = (p.out_rows + p.seg_rows - 1) / p.seg_rows;
    xp.f = p;
    if (with_blur) {
        // gray enters the vertical pass as an integer bit pattern (value q * 2^-149): the vertical
        // taps carry 2^75 and the horizontal taps 2^74 (powers of two: every rounding is unchanged)
        xp.gv0 = std::ldexp(g[0], 75); xp.gv1 = std::ldexp(g[1], 75); xp.gv2 = std::ldexp(g[2], 75);
        xp.gh0 = std::ldexp(g[0], 74); xp.gh1 = std::ldexp(g[1], 74); xp.gh2 = std::ldexp(g[2], 74);
        // S~ + 256 is rounded to a multiple of ulp = 2^-15 (error <= ulp/2).  A pixel whose 15 fraction
        // bits are >= a and <= 2^15 - 1 - a has frac(S~) in [(a - 1/2) ulp, 1 - (a + 1/2) ulp], i.e. S~ is
        // >= band away from an integer when a >= band / ulp + 1/2; all others are inside the guard band.
        // The bias carries the +a ulps (exact: a multiple of the ulp), so "inside" is "fraction bits < 2a" and
        // the masked value of such a pixel is the integer n it is close to; the reference's result is n or n - 1.
        const double ulp = std::ldexp(1.0, -kFracBits);
        const uint32_t a = (uint32_t)std::ceil(band / ulp + 0.5);
        xp.bias = (float)(256.0 + a * ulp);
        xp.zthr = (2u * a) << (32 - kFracBits);
        for (int i = 0; i < 25; i++) xp.fix.ws[i] = std::ldexp(p.w[i], 100);   // (exact: w >= 2^-70 or 0, checked in plan_weights_band)
        {   // (256 x 25 host operations: keep the last table)
            static std::mutex mu;
            static float last_w[25];
            static uint32_t last_tab[8];
            static bool have = false;
            std::lock_guard<std::mutex> lk(mu);
            if (!have || memcmp(last_w, p.w, sizeof(last_w)) != 0) {
                plan_flat_table(p.w, last_tab);
                memcpy(last_w, p.w, sizeof(last_w));
                have = true;
            }
            memcpy(xp.fix.flat_dec, last_tab, sizeof(last_tab));
        }
    }
    const long long blocks = (long long)n_frames * p.n_segs * p.n_band_groups;
    if (blocks <= 0 || blocks > 0x7fffffffLL) return fail(RIP_EINVAL, "rip_fused: grid of %lld blocks is out of range", blocks);
    const dim3 grid((unsigned)blocks);
    switch (fmt) {
    case RIP_FMT_RGB8:  launch_x2_t<NPX, 3, false>(with_blur, grid, s, xp); break;
    case RIP_FMT_BGR8:  launch_x2_t<NPX, 3, true>(with_blur, grid, s, xp); break;
    case RIP_FMT_RGBA8: launch_x2_t<NPX, 4, false>(with_blur, grid, s, xp); break;
    case RIP_FMT_BGRA8: launch_x2_t<NPX, 4, true>(with_blur, grid, s, xp); break;
    case RIP_FMT_GRAY8: case RIP_FMT_NV12: launch_x2_t<NPX, 1, false>(with_blur, grid, s, xp); break;
    default: return fail(RIP_EINVAL, "rip_fused: unsupported input format %d", fmt);
    }
    RIP_LAUNCH_CHECK();
    return RIP_OK;
}

// pixels per lane of the kernel that runs: RIP_FUSED_NPX = 8 | 4 (8 needs W % 8 == 0 and 8/16-byte aligned images)
static int x2_npx(int W, int cn, const uint8_t *d_in, const uint8_t *d_out)
{
    const int want = options().fused_npx == 4 ? 4 : 8;
    const uintptr_t in_align8 = cn == 4 ? 15u : 7u;   // (1 and 3 channels: 8 pixels are 8 / 24 bytes, loaded as 64-bit words)
    const bool ok8 = (W & 7) == 0 && !(reinterpret_cast<uintptr_t>(d_in) & in_align8) && !(reinterpret_cast<uintptr_t>(d_out) & 7u);
    if (want == 8 && ok8) return 8;
    return 4;  // fused_supported() already guarantees W % 4 == 0 and the 4-pixel alignments
}

int launch_fused(cudaStream_t s, const uint8_t *d_in, uint8_t *d_out, int W, int H, int n_frames, int fmt,
                 bool with_blur, const float *weights25, int in_row0, int in_rows, int out_row0, int out_rows,
                 int device)
{
    FusedParams p;
    memset(&p, 0, sizeof(p));
    p.in = d_in; p.out = d_out; p.W = W; p.H = H;
    p.in_row0 = in_row0; p.in_rows = in_rows; p.out_row0 = out_row0; p.out_rows = out_rows;
    p.slow_counter = g_slow_counter;
    double band = 0.0;
    float g[3] = {0.f, 0.f, 0.f};
    if (with_blur) {
        if (!plan_weights_band(weights25, g, &band))
            return fail(RIP_EUNSUPPORTED, "rip_fused: weights are not a non-negative symmetric separable 5x5 kernel");
        memcpy(p.w, weights25, sizeof(float) * 25);
    }
    const Format &f = *format_of(fmt);   // (fused_supported() checked the format)
    // whole NV12 frames carry their chroma plane behind the luma plane; row bands are passed as plain luma rows
    p.in_frame_bytes = (in_row0 == 0 && in_rows == H) ? frame_bytes(f, W, H) : (size_t)in_rows * W * f.channels;
    if (x2_npx(W, f.channels, d_in, d_out) == 8) return launch_fused_x2_n<8>(s, p, n_frames, fmt, with_blur, band, g, device);
    return launch_fused_x2_n<4>(s, p, n_frames, fmt, with_blur, band, g, device);
}

void fused_set_slow_counter(unsigned long long *d_counter) { g_slow_counter = d_counter; }

// ---------------------------------------------------------------------------------------------
// device self-test of the arithmetic shortcuts the fused kernel relies on, exhaustively:
// ---------------------------------------------------------------------------------------------
namespace {

// the x2 kernel's versions of the same two shortcuts: (1) sqrt.approx, then a multiply by 2^-149 (or
// 2^-127 on the 2^-22-scaled values of the no-blur variant) whose denormal result IS the rounded
// integer, then I2IP.U8.S32.SAT; (2) IDP.2A + FMUL2.RM / FFMA2.RP gray with the cold double evaluation.
__global__ void selftest_sqrt_x2_kernel(unsigned long long *bad)
{
    const unsigned m2_max = 2u * 1020u * 1020u;
    const float s44 = __uint_as_float((127u - 44u) << 23);  // 2^-44
    for (unsigned m2 = blockIdx.x * blockDim.x + threadIdx.x; m2 <= m2_max; m2 += gridDim.x * blockDim.x) {
        const unsigned want = (unsigned)min(__float2int_rn(__fsqrt_rn((float)m2)), 255);
        const u64 a = mul2(pk2(sqrt_approx((float)m2), sqrt_approx((float)m2 * s44)),
                           pk2(__uint_as_float(1u), __uint_as_float(0x00400000u)));
        const uint32_t packed = i2ip(hi2u(a), lo2u(a), 0u);
        if ((packed & 0xffu) != want || ((packed >> 8) & 0xffu) != want) atomicAdd(bad, 1ull);
    }
}

template <int NPX, int CN, bool BGR>
__global__ void selftest_gray_x2_kernel(unsigned long long *bad)
{
    constexpr int NP = NPX / 2, NW = NPX * CN / 4;
    // thread q handles triples NPX*q .. NPX*q + NPX-1 (triple i: c0 = i & 255, c1 = (i >> 8) & 255, c2 = i >> 16)
    for (unsigned q = blockIdx.x * blockDim.x + threadIdx.x; q < (1u << 24) / NPX; q += gridDim.x * blockDim.x) {
        uint8_t bytes[NW * 4];
#pragma unroll
        for (int j = 0; j < NPX; j++) {
            const unsigned i = NPX * q + j;
            bytes[CN * j + 0] = i & 255u; bytes[CN * j + 1] = (i >> 8) & 255u; bytes[CN * j + 2] = i >> 16;
            if (CN == 4) bytes[4 * j + 3] = (uint8_t)(i * 37u);  // alpha must be ignored
        }
        uint32_t w[NW];
#pragma unroll
        for (int k = 0; k < NW; k++)
            w[k] = bytes[4 * k] | (bytes[4 * k + 1] << 8) | (bytes[4 * k + 2] << 16) | ((uint32_t)bytes[4 * k + 3] << 24);
        u64 Q[NP], E[NP];
        const uint32_t any = gray_x2<NPX, CN, BGR>(w, Q, E);
        if (__any_sync(FULL, any & 1u)) {
            if (any & 1u) gray_fix_pairs<NPX, CN, BGR>(w, Q, E);
        }
#pragma unroll
        for (int j = 0; j < NPX; j++) {
            const unsigned i = NPX * q + j;
            const unsigned c0 = i & 255u, c1 = (i >> 8) & 255u, c2 = i >> 16;
            const unsigned want = BGR ? gray_exact(c2, c1, c0) : gray_exact(c0, c1, c2);
            const unsigned got = j < NP ? lo2u(Q[j % NP]) : hi2u(Q[j % NP]);
            if (got != want) atomicAdd(bad, 1ull);
        }
    }
}

}  // namespace

int fused_selftest(int device, unsigned long long *checked, unsigned long long *mismatches)
{
    unsigned long long *d_bad = nullptr;
    RIP_CUDA(cudaMalloc(&d_bad, sizeof(*d_bad)));
    RIP_CUDA(cudaMemset(d_bad, 0, sizeof(*d_bad)));
    const int grid = sm_count(device) * 8;
    selftest_sqrt_x2_kernel<<<grid, 256>>>(d_bad);
    selftest_gray_x2_kernel<8, 3, false><<<grid, 256>>>(d_bad);
    selftest_gray_x2_kernel<8, 3, true><<<grid, 256>>>(d_bad);
    selftest_gray_x2_kernel<8, 4, false><<<grid, 256>>>(d_bad);
    selftest_gray_x2_kernel<8, 4, true><<<grid, 256>>>(d_bad);
    selftest_gray_x2_kernel<4, 3, false><<<grid, 256>>>(d_bad);
    selftest_gray_x2_kernel<4, 3, true><<<grid, 256>>>(d_bad);
    selftest_gray_x2_kernel<4, 4, false><<<grid, 256>>>(d_bad);
    selftest_gray_x2_kernel<4, 4, true><<<grid, 256>>>(d_bad);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    unsigned long long bad = 0;
    if (e == cudaSuccess) e = cudaMemcpy(&bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost);
    cudaFree(d_bad);
    if (e != cudaSuccess) return cuda_fail(e, "fused_selftest", __FILE__, __LINE__);
    count_launch(9);
    *checked = 2ull * (2ull * 1020ull * 1020ull + 1ull) + 8ull * (1ull << 24);
    *mismatches = bad;
    return RIP_OK;
}

}  // namespace rip
