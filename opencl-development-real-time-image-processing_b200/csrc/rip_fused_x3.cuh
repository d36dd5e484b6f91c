// rip_fused_x3.cuh -- the production fused kernel: gray -> 5x5 Gaussian -> 3x3 Sobel (or gray -> Sobel) in
// one pass, written around what tools/pipe_probe.cu measured on B200 (profiles/r1_pipe_probe_*.txt):
//
//   pipe          lanes/clk/SM   used here for
//   FMA  (fp32)   128            FFMA2/FADD2/FMUL2 (two pixels per instruction: half the issue slots,
//                                same pipe time), scalar FADD for the halo taps, IDP.2A (64/clk)
//   ALU           64             LOP3, VIMNMX3, I2IP, SHF
//   XU            16             MUFU.SQRT only (I2F/F2I/FRND and IMAD.WIDE/.HI are slow: none on the hot path)
//   LSU/shuffle   32             LDG, SHFL, STS, STG
//
// Hot path (unchanged in substance since round 1, see DESIGN.md 3.1):
//   * gray: t = 299r+587g+114b by IDP.2A; the INTEGER bit pattern of t, read as a float, is the denormal
//     t*2^-149, so floor(t/1000) is ONE multiply rounded toward -inf by the float just above 1/1000
//     (FMUL2.RM), and its result is again an integer bit pattern that feeds the blur's FFMAs directly.
//     A second FMA rounded toward +inf with the float just below 1/1000 yields 1 exactly on the multiples
//     of 1000, the only triples where the reference's double arithmetic (Comparator.cpp:41) can land one
//     below t/1000.
//   * blur: separable fp32 fast path; S~ + bias (bias = 256 + a ulps, a = guard band in ulps of 2^-15) puts
//     floor(S~) in mantissa bits 15..22 and the fraction in bits 0..14; a pixel is inside the guard band iff
//     its fraction bits are below 2a (one shift + half a VIMNMX3 per pixel), and then the masked value is
//     n = the integer S~ is close to; the reference's result is n or n - 1.
//   * Sobel on the biased values 256+b (all sums exact in fp32); round-half-even + saturation = FMUL2 by
//     2^-149 + I2IP.U8.S32.SAT; one predicated 64-bit store per lane per row.
//   * a lane owns NPX adjacent pixels, pixel j paired with pixel j+NPX/2 in one 64-bit register so that every
//     horizontal tap of a pair is again an aligned pair; the few taps that straddle a lane boundary are formed
//     with scalar FADDs written straight into the halves of the result pair (no pair construction, no moves).
//
// Round 2: the cold paths.  Round 1 handled a guard-band pixel warp-cooperatively, one pixel at a time, and
// patched a shared-memory copy that the hot path re-read with predicated loads: flat content (every pixel in
// the band) ran 77x slower than textured content, black 21x.  Now:
//   * both cold paths are LANE-PARALLEL and return one 8-bit DECREMENT MASK per lane; the hot registers are
//     touched only by an in-place "subtract the mask bit" block inside the cold branch (no predicated reloads,
//     no copies of the hot values, nothing of the cold path on the hot instruction stream).
//   * gray fix: the flagged pixel's reference expression is simply evaluated in double (DMUL/DADD, B200 has
//     full-rate-enough FP64 for a path that runs on 0.1 % of the pixels): no lookup table, no table copy per
//     block, no shared memory for it.
//   * blur fix: (1) a lane whose whole 5 x (NPX+4) neighbourhood in the gray ring is one value v takes all its
//     pixels from a 256-bit table (bit v = "the reference's sum of a constant window v truncates below v'"),
//     evaluated on the host with the reference's own sequence for the weights in use: flat, black, clipped and
//     letterboxed content costs one table lookup per lane-row; (2) otherwise each flagged pixel is replayed by
//     ITS lane with the reference's exact ky-major / kx-minor sequence from the ring, all flagged lanes at once.
//
// Included by rip_fused.cu inside its anonymous namespace.

typedef unsigned long long u64;

__device__ __forceinline__ u64 pk2(float lo, float hi) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ u64 pk2u(uint32_t lo, uint32_t hi) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi)); return r; }
__device__ __forceinline__ float lo2(u64 v) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); return lo; }
__device__ __forceinline__ float hi2(u64 v) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); return hi; }
__device__ __forceinline__ uint32_t lo2u(u64 v) { uint32_t lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v)); return lo; }
__device__ __forceinline__ uint32_t hi2u(u64 v) { uint32_t lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v)); return hi; }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) { u64 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 add2(u64 a, u64 b) { u64 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 sub2(u64 a, u64 b) { u64 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 mul2_rm(u64 a, u64 b) { u64 d; asm("mul.rm.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 fma2_rp(u64 a, u64 b, u64 c) { u64 d; asm("fma.rp.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
// d = (c & 0xffff) << 16 | sat_u8(a) << 8 | sat_u8(b)
__device__ __forceinline__ uint32_t i2ip(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

constexpr float kInvK_up = 1.0000000474974513e-3f;   // 0x3A83126F: the float just ABOVE 1/1000
constexpr float kInvK_dn = 9.9999993108212948e-4f;   // 0x3A83126E: the float just BELOW 1/1000
constexpr float kBias = 256.0f;                      // [256, 512): ulp 2^-15, floor(S~) in mantissa bits 15..22
constexpr uint32_t kBiasMask = 0xffff8000u;
constexpr int kFracBits = 15;

// what the out-of-line blur fix reads (it gets a pointer to this part of the kernel parameters)
struct BlurFixConst {
    float ws[25];          // the exact 2-D weights times 2^100 (for the replay: products stay normal, see blur_replay_lane)
    uint32_t flat_dec[8];  // bit v: a constant 5x5 window of gray v gives the reference sum S with trunc(S) = rint(S) - 1
};

struct X2Params {
    FusedParams f;
    float gv0, gv1, gv2;   // vertical taps   * 2^75  (gray enters as the integer bit pattern q = q * 2^-149)
    float gh0, gh1, gh2;   // horizontal taps * 2^74
    float bias;            // kBias + a * 2^-15: the guard band's lower edge rides in the bias, so that
    uint32_t zthr;         // a pixel is inside the band iff (bits << 17) < zthr = 2a << 17, and its masked value is then n
    BlurFixConst fix;
};

// ---- exact gray of NPX packed pixels -> NPX/2 pairs of integer bit patterns ---------------------
// returns the OR of the "t is a multiple of 1000" flags in bit 0
template <int NPX, int CN, bool BGR>
__device__ __forceinline__ uint32_t gray_x2(const uint32_t *w, u64 *Q, u64 *E)
{
    constexpr int NP = NPX / 2;
    if constexpr (CN == 1) {
        // the input IS the gray image (GRAY8, or the luma plane of NV12): isolate the bytes; an isolated byte is
        // already the integer bit pattern the later stages consume.  No exactness cases here.
#pragma unroll
        for (int j = 0; j < NP; j++) {
            Q[j] = pk2u(__byte_perm(w[j / 4], 0u, 0x4440u | (uint32_t)(j & 3)), __byte_perm(w[(j + NP) / 4], 0u, 0x4440u | (uint32_t)((j + NP) & 3)));
            E[j] = 0ull;
        }
        return 0u;
    } else {
    constexpr uint32_t cA = BGR ? 114u : 299u, cB = 587u, cC = BGR ? 299u : 114u;  // weights of byte 0,1,2
    constexpr uint32_t AB = cA | (cB << 16), C0 = cC, zA = cA << 16, BC = cB | (cC << 16);
    uint32_t t[NPX];
#pragma unroll
    for (int g = 0; g < NPX / 4; g++) {
        const uint32_t *v = w + g * CN;
        if constexpr (CN == 4) {
#pragma unroll
            for (int j = 0; j < 4; j++) t[4 * g + j] = __dp2a_hi(C0, v[j], __dp2a_lo(AB, v[j], 0u));  // alpha x 0
        } else {
            // byte stream: p0 = v0.b0-2, p1 = v0.b3 v1.b0-1, p2 = v1.b2-3 v2.b0, p3 = v2.b1-3
            t[4 * g + 0] = __dp2a_hi(C0, v[0], __dp2a_lo(AB, v[0], 0u));
            t[4 * g + 1] = __dp2a_lo(BC, v[1], __dp2a_hi(zA, v[0], 0u));
            t[4 * g + 2] = __dp2a_lo(C0, v[2], __dp2a_hi(AB, v[1], 0u));
            t[4 * g + 3] = __dp2a_hi(BC, v[2], __dp2a_lo(zA, v[2], 0u));
        }
    }
    const u64 up = pk2(kInvK_up, kInvK_up), ndn = pk2(-kInvK_dn, -kInvK_dn);
    uint32_t any = 0;
#pragma unroll
    for (int j = 0; j < NP; j++) {
        const u64 T = pk2u(t[j], t[j + NP]);
        Q[j] = mul2_rm(T, up);        // floor(t * up) = floor(t / 1000)          (t <= 255000)
        E[j] = fma2_rp(T, ndn, Q[j]); // ceil(q - t * dn): 1 iff t = 1000 q > 0, else -0 / +0
        any |= lo2u(E[j]) | hi2u(E[j]);
    }
    return any;
    }
}

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }
__device__ __forceinline__ float lds_f32(uint32_t addr) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr)); return v; }
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_b64(uint32_t addr, u64 v) { asm volatile("st.shared.b64 [%0], %1;" ::"r"(addr), "l"(v) : "memory"); }
__device__ __forceinline__ uint32_t lds_u8(uint32_t addr) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }

// ---- the gray ring ------------------------------------------------------------------------------------------------
// Every warp keeps the last kRing = 6 gray rows of its band in shared memory, as integer bit patterns (= q * 2^-149 read
// as floats).  Only the cold paths read it: the constant-window test and the exact replay of guard-band pixels (the
// vertical blur pass of the hot path carries its partial sums in registers, WarpX).  Layout of a row (kRowB = 128 * NPX
// bytes): NP/2 planes of 512 bytes; plane p holds, for lane L at byte 16 L, the pairs 2p and 2p+1 of that lane (pair k =
// (pixel k, pixel k + NP)): a lane stores and reloads its row with NP/2 conflict-free 128-bit accesses.
constexpr int kRing = 6;

// byte offset inside a ring row of band column c (column 0 = pixel 0 of lane 0)
template <int NPX>
__device__ __forceinline__ uint32_t ring_off(uint32_t c)
{
    constexpr uint32_t NP = NPX / 2;
    const uint32_t L = c / NPX, j = c % NPX, pr = j % NP, h = j / NP;
    return (pr / 2u) * 512u + L * 16u + (pr % 2u) * 8u + h * 4u;
}

// ---- cold, lane-parallel: the exact gray of pixels whose t = 299r+587g+114b is a multiple of 1000 -----------------------------
// c_gray_down: bit (r | g << 8) = "the reference's double expression (Comparator.cpp:41) lands one below t/1000" for the one b
// that makes t a multiple of 1000 with this (r, g) (tools/make_gray_table.py evaluates the reference expression itself; the
// device self-test checks all 2^24 triples against a double evaluation).  An initialised __constant__ array: part of the module
// image, nothing to copy or order at run time.
__constant__ uint32_t c_gray_down[2048] = {
#include "rip_gray_table.inc"
};

// bit 0 of the result: table bit of pixel j of the lane (bytes of the pixel at compile-time positions of the raw words)
template <int CN, bool BGR>
__device__ __forceinline__ uint32_t gray_down_bit(const uint32_t *w, int j)
{
    const int o = CN * j + (BGR ? 1 : 0), a = o / 4, s = o % 4;   // the key's two bytes start at byte o of the lane's raw bytes: (r, g) or, for BGR, (g, r)
    uint32_t key;   // r | g << 8 in the low 16 bits, anything above
    if (!BGR) {
        key = s == 0 ? w[a] : s <= 2 ? w[a] >> (8 * s) : __funnelshift_r(w[a], w[a + 1], 24);
    } else {        // bytes (g, r) -> (r, g)
        key = s <= 2 ? __byte_perm(w[a], 0u, (uint32_t)((s + 1) | (s << 4))) : __byte_perm(w[a], w[a + 1], 0x34u);
    }
    const uint32_t word = c_gray_down[(key >> 5) & 2047u];
    return word >> (key & 31u);
}

// Every half of E (gray_x2) is 1 (t is a multiple of 1000), +0 or -0.  Pair by pair: where a half is flagged, subtract the table
// bit of that pixel.  Everything sits at compile-time positions: no pixel index at run time, no staging in shared memory, no
// loop -- one flagged pixel costs the four pair tests and one 14-instruction block (round 2's first version staged the raw
// bytes in shared memory, looped over a bit mask and evaluated the double expression: ~95 warp instructions per excursion,
// and an excursion costs its instruction count times the ~6 cycles between two issues of one warp).
template <int NPX, int CN, bool BGR>
__device__ __forceinline__ void gray_fix_pairs(const uint32_t *w, u64 *Q, const u64 *E)
{
    constexpr int NP = NPX / 2, NW = NPX * CN / 4;
    // constant regions first (every grey / white / clipped pixel has t = 1000 v, so flat content enters here on every row):
    // all raw words equal -- and r = g = b for 3-byte pixels -- means one colour, one table bit for the lane
    uint32_t diff = 0;
#pragma unroll
    for (int k = 1; k < NW; k++) diff |= w[k] ^ w[0];
    if (CN == 3) diff |= w[0] ^ __byte_perm(w[0], 0u, 0x2103);
    if (diff == 0u) {
        const uint32_t sub = gray_down_bit<CN, BGR>(w, 0) & lo2u(E[0]) & 1u;
#pragma unroll
        for (int k = 0; k < NP; k++) Q[k] = pk2u(lo2u(Q[k]) - sub, hi2u(Q[k]) - sub);
        return;
    }
#pragma unroll
    for (int k = 0; k < NP; k++) {
        const uint32_t el = lo2u(E[k]), eh = hi2u(E[k]);
        if ((el | eh) & 1u) {
            const uint32_t ql = lo2u(Q[k]) - (gray_down_bit<CN, BGR>(w, k) & el & 1u);
            const uint32_t qh = hi2u(Q[k]) - (gray_down_bit<CN, BGR>(w, k + NP) & eh & 1u);
            Q[k] = pk2u(ql, qh);
        }
    }
}

// in place: pixel j of the lane -= bit j of `dec`, on integer bit patterns (gray) or, scaled by 2^15, on the biased
// floats of the blur stage (256 + b with ulp 2^-15: one integer step of the value is 0x8000 in the bit pattern)
template <int NPX, int SHIFT>
__device__ __forceinline__ void apply_dec(u64 *V, uint32_t dec)
{
    constexpr int NP = NPX / 2;
#pragma unroll
    for (int j = 0; j < NP; j++) {
        const uint32_t lo = lo2u(V[j]) - (((dec >> j) & 1u) << SHIFT);
        const uint32_t hi = hi2u(V[j]) - (((dec >> (j + NP)) & 1u) << SHIFT);
        V[j] = pk2u(lo, hi);
    }
}

// this lane's raw bytes of one input row
template <int NPX, int CN>
struct RawX {
    uint32_t w[NPX * CN / 4];
};

// Input rows travel global -> shared with cp.async, NB rows ahead of their use (one commit group per row, the step of row r
// waits until at most NB - 1 groups are pending), and each lane reads its own bytes back with LDS.  Rounds 1-2 used register
// loads NB rows ahead: the first consumer of a loaded row in ONE of the unrolled steps then held 8.5 % of the kernel's stall
// samples (profiles/r2m_fused_x3_hotspots.txt) whatever the distance -- a wait on a load's scoreboard also waits for every
// younger load that shares it (seen and fixed first in the streaming blur, rip_blur_stream.cuh) -- and the three row buffers
// occupied 18 registers.  Lanes outside the image fetch the start of the row (their pointer has x offset 0); their pixels are
// never consumed.

// this lane's NW words of a row: global -> shared (asynchronous), shared -> registers
template <int NPX, int CN>
__device__ __forceinline__ void cp_row_x3(uint32_t dst, const uint8_t *p)
{
    constexpr int NW = NPX * CN / 4;
    if constexpr (NW == 1) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(p) : "memory");
    } else if constexpr (NW == 2) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(p) : "memory");
    } else if constexpr (NW == 3) {
#pragma unroll
        for (int k = 0; k < 3; k++) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4u * k), "l"(p + 4 * k) : "memory");
    } else if constexpr (NW == 4) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(p) : "memory");
    } else if constexpr (NW == 6) {
#pragma unroll
        for (int k = 0; k < 3; k++) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + 8u * k), "l"(p + 8 * k) : "memory");
    } else {
#pragma unroll
        for (int k = 0; k < 2; k++) asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * k), "l"(p + 16 * k) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}

template <int NPX, int CN>
__device__ __forceinline__ void lds_row_x3(RawX<NPX, CN> &r, uint32_t a)
{
    constexpr int NW = NPX * CN / 4;
    if constexpr (NW == 1) {
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r.w[0]) : "r"(a) : "memory");
    } else if constexpr (NW == 2) {
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(r.w[0]), "=r"(r.w[1]) : "r"(a) : "memory");
    } else if constexpr (NW == 3) {
#pragma unroll
        for (int k = 0; k < 3; k++) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r.w[k]) : "r"(a + 4u * k) : "memory");
    } else if constexpr (NW == 4) {
        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.w[0]), "=r"(r.w[1]), "=r"(r.w[2]), "=r"(r.w[3]) : "r"(a) : "memory");
    } else if constexpr (NW == 6) {
#pragma unroll
        for (int k = 0; k < 3; k++) asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(r.w[2 * k]), "=r"(r.w[2 * k + 1]) : "r"(a + 8u * k) : "memory");
    } else {
#pragma unroll
        for (int k = 0; k < 2; k++)
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.w[4 * k]), "=r"(r.w[4 * k + 1]), "=r"(r.w[4 * k + 2]), "=r"(r.w[4 * k + 3]) : "r"(a + 16u * k) : "memory");
    }
}

// The vertical blur pass carries four rows of partial sums in registers (accumulate form, five packed FMAs per pixel pair and
// row, no shared-memory reads on the hot path).  Re-reading gray rows r-1 .. r-4 from the ring instead (eight LDS.128 per lane
// and row, 32 registers of state less) was measured on 32 4K frames with the round's final cold paths: 436 us against 418 us
// (114 against 122 registers, both four blocks per SM, neither spills).
template <int NPX, int CN>
struct WarpX {
    u64 a0[NPX / 2], a1[NPX / 2], a2[NPX / 2], a3[NPX / 2];  // pending vertical sums of blurred rows r-2 .. r+1
    u64 F1[NPX / 2], F2[NPX / 2];   // rows yb-1 and yb-2 of the image the Sobel stage reads
};

struct GeoX {
    const uint8_t *src;      // this lane's pixels in the input row that was loaded last
    uint8_t *dst;            // this lane's pixels in the output row produced next
    uint32_t ring_lane;      // shared-memory byte address of this lane's 16 bytes in plane 0 of slot 0 of the warp's gray ring
    uint32_t ringA, ringB;   // main loop: ring_lane + the half (slots 0-2 / 3-5) this trip writes / wrote last trip
    uint32_t slot;           // head / tail rows: slot of the newest gray row
    uint32_t raw_lane, rs;   // shared-memory byte address of this lane's bytes in slot 0 of the warp's raw-row ring; head / tail rows: slot of the row in use
    uint32_t in_pitch;
    int adv_lo, adv_n;       // the source pointer advances before the load of step r iff 0 <= r - adv_lo < adv_n
    int lane;
    uint32_t need;           // pixels of this lane whose blurred value feeds an output (bit j = pixel j): all of lanes 1..30,
                             // only the pixel next to the band in the two halo lanes, none in lanes outside the image
    bool e_left, e_right;    // this lane holds image column 0 / W-1 (border rules in x apply to it)
    bool edge_warp;          // warp-uniform: some lane of this warp has e_left or e_right set (2 of the 16 bands of a 4K row)
    uint32_t store_lane;
    int r_store, r_last;     // first / last step that produces an output row
};

// ---- cold, lane-parallel: the exact blurred value of guard-band pixels ---------------------------------------------
// Both functions run in every flagged lane at once; lanes do not cooperate, so there is no warp-level synchronisation
// inside (the caller's __syncwarp made the newest ring row visible).  `ring0` = address of slot 0 of the warp's ring
// (lane 0), `newest` = slot of gray row r; the 5x5 windows span rows r-4 .. r.  With S = the reference's sum
// (GaussianBlur.cpp:236-258) and n = rint(S) -- the fast path's value of a guard-band pixel, see the file header -- the
// reference's result trunc(S) is n - 1 iff S < n; both functions answer that question.

// (1) constant neighbourhood: if the 5 rows x (NPX + 4) columns around the lane's pixels all hold one gray value v, every
// 5x5 window of the lane is that constant and the answer is bit v of xp.flat_dec, which the host evaluated with the
// reference's own sequence for the weights in use.  Returns 0 / 1 = the answer, 2 = the neighbourhood is not constant.
// `hist` (one word per lane in shared memory: a register that lives across the row loop costs the hot path 16 moves per trip, measured)
// remembers the last row at which this test found the lane's 12 columns of the NEWEST ring row constant, the
// value, and for how many consecutive rows that has held (row << 12 | run << 8 | value): inside a constant region the test then
// reads one ring row per image row instead of five (flat content: 945 -> see profiles/README.md).  A row that did not come
// through here breaks the run (its row number is missing), so the history never claims more than was checked.
// Per-lane table in shared memory, filled once per block (fused_x2_kernel): words 0 .. NPX+3 = byte offset, relative to the lane's
// own 16 bytes in plane 0 of a ring row, of the ring word of the pixel `rel - 2` columns from the lane's first pixel, with the
// clamp-to-edge rule of the lane that holds an image border already applied (GaussianBlur.cpp:240); word 15 = `hist`.  The cold
// paths read their column offsets from here: no constant-memory look-ups, no min / max, no border branch in the row bodies (the
// main loop holds three copies of every cold block, and its size costs time even when the blocks never run).
constexpr int kLaneTabWords = 16;
__shared__ uint32_t s_lane_tab[kWarpsPerBlock * 32 * kLaneTabWords];

template <int NPX>
__device__ __forceinline__ uint32_t blur_flat_lane(uint32_t ring_lane, uint32_t newest, uint32_t tab, const uint32_t *flat_dec, int r)
{
    constexpr uint32_t kRowB = 32 * NPX * 4;
    const uint32_t ol2 = lds_u32(tab), ol1 = lds_u32(tab + 4u), or0 = lds_u32(tab + 4u * (NPX + 2)), or1 = lds_u32(tab + 4u * (NPX + 3));
    const uint32_t hist_addr = tab + 4u * (kLaneTabWords - 1);
    const uint32_t v = lds_u32(ring_lane + newest * kRowB);
    // do the lane's NPX + 4 columns of the ring row at `row` (this lane's plane-0 address) all hold v?  (0 = yes)
    auto row_diff = [&](uint32_t row) -> uint32_t {
        uint32_t diff = 0;
#pragma unroll
        for (int pl = 0; pl < NPX / 4; pl++) {
            uint32_t a, b, c, d;
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(row + 512 * pl));
            diff |= (a ^ v) | (b ^ v);
            diff |= (c ^ v) | (d ^ v);
        }
        diff |= (lds_u32(row + ol2) ^ v) | (lds_u32(row + ol1) ^ v);
        diff |= (lds_u32(row + or0) ^ v) | (lds_u32(row + or1) ^ v);
        return diff;
    };
    const uint32_t rr = (uint32_t)r & 0xfffffu, prev = (uint32_t)(r - 1) & 0xfffffu;
    const uint32_t hist = lds_u32(hist_addr);
    const uint32_t known = ((hist >> 12) == prev && (hist & 0xffu) == v) ? ((hist >> 8) & 15u) : 0u;   // rows r-1 .. r-known are constant v
    // row r, then the rows nobody has looked at yet: r-known-1 .. r-4 (only at the first rows of a constant region)
    uint32_t k = 0u, new_hist = 0u, ans = 2u;
#pragma unroll 1
    for (;;) {
        const uint32_t s = newest >= k ? newest - k : newest + (uint32_t)kRing - k;
        if (row_diff(ring_lane + s * kRowB)) {
            if (k) new_hist = rr << 12 | k << 8 | v;   // rows r .. r-k+1 are constant
            break;
        }
        k = k == 0u ? known + 1u : k + 1u;
        if (k >= 5u) {
            const uint32_t rows_ok = known >= 4u ? known + 1u : 5u;   // consecutive constant rows ending at row r
            new_hist = rr << 12 | (rows_ok > 8u ? 8u : rows_ok) << 8 | v;
            ans = (flat_dec[v >> 5] >> (v & 31u)) & 1u;
            break;
        }
    }
    sts_u32(hist_addr, new_hist);
    return ans;
}

// byte offset, relative to the lane's own 16 bytes in plane 0, of the ring word of the pixel `rel - 2` columns from
// the lane's first pixel (rel in [0, NPX + 4): two pixels of the lane to the left .. two of the lane to the right)
template <int NPX>
struct RingRel {
    int v[NPX + 4];
    constexpr RingRel() : v()
    {
        for (int rel = 0; rel < NPX + 4; rel++) {
            int c = rel - 2, dl = 0;
            if (c < 0) { c += NPX; dl = -1; }
            if (c >= NPX) { c -= NPX; dl = 1; }
            const int pr = c % (NPX / 2), h = c / (NPX / 2);
            v[rel] = dl * 16 + (pr / 2) * 512 + (pr % 2) * 8 + h * 4;
        }
    }
};
__constant__ RingRel<8> c_ring_rel8;
__constant__ RingRel<4> c_ring_rel4;

// (2) the reference's 25-tap sequence for each of the pixels in `my` (bit j = pixel j); returns the mask of those whose
// result is n - 1.  The ring holds gray as integer bit patterns (= q * 2^-149 as floats) and ws the weights times
// 2^100: fl(q*2^-149 * w*2^100) = fl(q * w) * 2^-49 exactly (same mantissa, results stay normal), likewise every partial
// sum, so the scaled chain rounds exactly like the reference's (ky-major / kx-minor from 0.0f, unfused) and needs no
// integer-to-float conversion.  `rowaddr[i]` = shared-memory address of this lane's 16 bytes (plane 0) of gray row r - i;
// in the main loop those are compile-time offsets from two registers, so the 25 loads need ten address adds.  The column
// offsets come from the lane's table (s_lane_tab), clamp-to-edge included.
// What an excursion costs is its executed instruction count (the kernel's time is its warp-instruction count at a steady
// ~65 % issue rate, profiles/README.md), so everything that is not the 25 loads, 25 products and 25 adds is kept short.
// (Out of line -- one __noinline__ copy for all row bodies, main loop 1126 instead of 1693 instructions -- was measured:
// 445 us against 431 us; the call sequence and the run-time ring slots cost more than the smaller loop gains.)
template <int NPX>
__device__ __forceinline__ uint32_t blur_replay_lane(uint32_t my, const uint32_t (&rowaddr)[5], uint32_t tab, const BlurFixConst &cst)
{
    uint32_t dec = 0;
#pragma unroll 1
    while (my) {
        const uint32_t j = (uint32_t)__ffs(my) - 1u;
        my &= my - 1u;
        uint32_t off[5];
#pragma unroll
        for (int kx = 0; kx < 5; kx++) off[kx] = lds_u32(tab + 4u * j + 4u * kx);   // columns j-2 .. j+2 of the lane, clamped to the image
        float g25[25];
#pragma unroll
        for (int ky = 0; ky < 5; ky++)
#pragma unroll
            for (int kx = 0; kx < 5; kx++) g25[ky * 5 + kx] = __uint_as_float(lds_u32(rowaddr[4 - ky] + off[kx]));
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < 25; t++) acc = __fadd_rn(acc, __fmul_rn(g25[t], cst.ws[t]));
        acc = __fmul_rn(acc, 562949953421312.0f);   // * 2^49: back to the reference's scale (exact)
        dec |= (acc < rintf(acc) ? 1u : 0u) << j;
    }
    return dec;
}

// One image row of the sliding window: consumes input row r (clamped to the rows of the band) from the raw-ring slot at
// `raw_addr`, where it was fetched NB steps earlier, fetches row r + NB into the same slot, and -- for r_store <= r <= r_last --
// stores output row r - HALO.  The border rules are applied at run time (per-lane selects in x, two rare uniform branches in
// y), so this is the only copy of the row body; the caller's main loop unrolls it by NB, which makes the two-row Sobel delay
// line register renames.
// What a copy of the row body has to check at run time:
//   SPECIAL  head and tail rows of a segment: does this row store, does the next input row exist, BORDER_REFLECT_101 in y.
//            The main loop's copies check none of that.
//   KS       position of the row inside a main-loop trip (0, 1, 2): the ring slots of rows r .. r-4 are then compile-time
//            offsets from the two half-ring bases geo.ringA / geo.ringB.  KS = -1 (head / tail rows): run-time slots.
// Every copy takes the per-lane border selects in x behind one warp-uniform branch (geo.edge_warp: the band holds image
// column 0 and/or W-1).
template <int NPX, int CN, bool BGR, bool BLUR, bool SPECIAL, bool STATS, int KS, int NB>
__device__ __forceinline__ void step_x2(WarpX<NPX, CN> &st, const uint32_t raw_addr, const X2Params &xp, GeoX &geo, int r)
{
    RawX<NPX, CN> buf;   // row r: fetched NB steps ago
    asm volatile("cp.async.wait_group %0;" ::"n"(NB - 1) : "memory");
    lds_row_x3<NPX, CN>(buf, raw_addr);
    constexpr int NP = NPX / 2;
    constexpr int kRowB = 32 * NPX * 4;  // bytes per ring row
    static_assert(SPECIAL == (KS < 0), "head / tail rows use run-time ring slots");
    const FusedParams &p = xp.f;
    const int W = p.W, H = p.H;
    (void)H;

    // ---- 1. gray of row r; fetch row r + NB --------------------------------------------------------
    u64 Q[NP];
    uint32_t rowaddr[5];   // this lane's 16 bytes (plane 0) of the ring rows holding gray rows r, r-1, .. r-4
    {
        u64 E[NP];
        const uint32_t flagged = gray_x2<NPX, CN, BGR>(buf.w, Q, E) & 1u;
        if (CN != 1 && __builtin_expect(__any_sync(FULL, flagged), 0)) {
            if (flagged) gray_fix_pairs<NPX, CN, BGR>(buf.w, Q, E);
        }
        if constexpr (BLUR) {
            // park the integer gray row in the shared ring (the blur's cold paths of this and the next four rows read it
            // back); rows r-1 .. r-4 sit in the slots before it
            if constexpr (KS < 0) {
                geo.slot = geo.slot == (uint32_t)kRing - 1u ? 0u : geo.slot + 1u;
                uint32_t s4 = geo.slot;
#pragma unroll
                for (int i = 0; i < 5; i++) {
                    rowaddr[i] = geo.ring_lane + s4 * kRowB;
                    s4 = s4 == 0u ? (uint32_t)kRing - 1u : s4 - 1u;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 5; i++) {
                    const int v = KS - i;   // slot relative to this trip's half: negative = the half written one trip (or, for -4, two trips) ago
                    rowaddr[i] = v >= 0 ? geo.ringA + v * kRowB : v >= -3 ? geo.ringB + (v + 3) * kRowB : geo.ringA + (v + 6) * kRowB;
                }
            }
#pragma unroll
            for (int pl = 0; pl < NP / 2; pl++)
                asm volatile("st.shared.v2.b64 [%0], {%1, %2};" ::"r"(rowaddr[0] + 512 * pl), "l"(Q[2 * pl]), "l"(Q[2 * pl + 1]) : "memory");
        }
        if constexpr (SPECIAL) {
            if ((unsigned)(r - geo.adv_lo) < (unsigned)geo.adv_n) geo.src += geo.in_pitch;
        } else {
            geo.src += geo.in_pitch;   // (the main loop stops short of the rows where the band ends)
        }
        cp_row_x3<NPX, CN>(raw_addr, geo.src);   // row r + NB into the slot row r just left
    }

    // F[j] = (f[j], f[j + NP]): the row the Sobel stage consumes (blurred row yb, biased by kBias, or
    // the gray row scaled to normal floats when there is no blur stage)
    u64 F[NP];
    const int yb = BLUR ? r - 2 : r;
    if constexpr (BLUR) {
        const u64 GV0 = pk2(xp.gv0, xp.gv0), GV1 = pk2(xp.gv1, xp.gv1), GV2 = pk2(xp.gv2, xp.gv2);
        u64 V[NP];
        // vertical pass, accumulate form: row r completes blurred row r-2
#pragma unroll
        for (int j = 0; j < NP; j++) {
            V[j] = fma2(GV2, Q[j], st.a0[j]);
            st.a0[j] = fma2(GV1, Q[j], st.a1[j]);
            st.a1[j] = fma2(GV0, Q[j], st.a2[j]);
            st.a2[j] = fma2(GV1, Q[j], st.a3[j]);
            st.a3[j] = mul2(GV2, Q[j]);
        }
        if constexpr (SPECIAL) {
            // warm-up rows of a segment: the first blurred row any stored output reads (ys - 1) completes at step
            // r_store - 2; before that only the gray ring is filled (the vote tells the compiler that the whole
            // warp leaves together)
            if (__all_sync(FULL, r < geo.r_store - 2)) {
                geo.dst += W;
                return;
            }
        }
        // horizontal pass.  c[m] = V of pixel m (pixel m lives in pair m % NP, half m / NP); e2 = c[m-2] + c[m+2],
        // e1 = c[m-1] + c[m+1].  Clamp-to-edge columns (GaussianBlur.cpp:240): V is linear in the gray column, so the
        // clamp applies to V: left of column 0 / right of column W-1 repeat it.
        float Vm2 = __shfl_up_sync(FULL, hi2(V[NP - 2]), 1), Vm1 = __shfl_up_sync(FULL, hi2(V[NP - 1]), 1);
        float Vp0 = __shfl_down_sync(FULL, lo2(V[0]), 1), Vp1 = __shfl_down_sync(FULL, lo2(V[1]), 1);
        if (geo.edge_warp) {   // (interior bands skip the selects where ptxas keeps the branch)
            Vm2 = geo.e_left ? lo2(V[0]) : Vm2;
            Vm1 = geo.e_left ? lo2(V[0]) : Vm1;
            Vp0 = geo.e_right ? hi2(V[NP - 1]) : Vp0;
            Vp1 = geo.e_right ? hi2(V[NP - 1]) : Vp1;
        }
        // value of pixel m of this lane, m in [-2, NPX+2)
        auto c = [&](int m) -> float {
            if (m == -2) return Vm2;
            if (m == -1) return Vm1;
            if (m == NPX) return Vp0;
            if (m == NPX + 1) return Vp1;
            return m < NP ? lo2(V[m]) : hi2(V[m - NP]);
        };
        const u64 GH0 = pk2(xp.gh0, xp.gh0), GH1 = pk2(xp.gh1, xp.gh1), GH2 = pk2(xp.gh2, xp.gh2);
        const u64 BIAS = pk2(xp.bias, xp.bias);
#pragma unroll
        for (int j = 0; j < NP; j++) {
            // pairs (j, j+NP): taps at distance d are the pairs (j+d, j+NP+d) -- aligned pairs V[j+d] while both
            // halves stay inside the lane; otherwise two scalar adds written straight into the halves of the result
            u64 e2, e1;
            if (j - 2 >= 0 && j + 2 < NP) e2 = add2(V[j - 2], V[j + 2]);
            else e2 = pk2(__fadd_rn(c(j - 2), c(j + 2)), __fadd_rn(c(j + NP - 2), c(j + NP + 2)));
            if (j - 1 >= 0 && j + 1 < NP) e1 = add2(V[j - 1], V[j + 1]);
            else e1 = pk2(__fadd_rn(c(j - 1), c(j + 1)), __fadd_rn(c(j + NP - 1), c(j + NP + 1)));
            // S~ of pixels j, j + NP, plus the bias (it rides in the FMA chain): floor(S~) in bits 15..22, fraction below
            F[j] = fma2(GH2, e2, fma2(GH1, e1, fma2(GH0, V[j], BIAS)));
        }
        // guard band: fraction bits below 2a (the bias carries +a ulps)
        uint32_t zmin = 0xffffffffu;
#pragma unroll
        for (int j = 0; j < NP; j++)
            zmin = __vimin3_u32(zmin, lo2u(F[j]) << (32 - kFracBits), hi2u(F[j]) << (32 - kFracBits));
        const uint32_t flagged = zmin < xp.zthr ? 1u : 0u;
        if (__builtin_expect(__any_sync(FULL, flagged), 0)) {
            __syncwarp();  // the newest ring row was just stored by the other lanes
            if (flagged) {
                // Which pixels are inside the band and feed an output?  A pixel whose masked value is n = 0 needs no fix at all: the
                // reference's result is n or n - 1 and cannot be negative (black bars and frames leave here).
                const uint32_t zero_bits = __float_as_uint(kBias);
                const uint32_t tab = (uint32_t)__cvta_generic_to_shared(&s_lane_tab[threadIdx.x * kLaneTabWords]);
                uint32_t my = 0, dec = 2u;
#pragma unroll
                for (int j = 0; j < NP; j++) {
                    const uint32_t l = lo2u(F[j]), h = hi2u(F[j]);
                    my |= (((l << (32 - kFracBits)) < xp.zthr && (l & kBiasMask) != zero_bits) ? 1u : 0u) << j;
                    my |= (((h << (32 - kFracBits)) < xp.zthr && (h & kBiasMask) != zero_bits) ? 1u : 0u) << (j + NP);
                }
                my &= geo.need;
                // Constant regions: every pixel of the lane is inside the band and the fast path's values are bit-identical (a cheap
                // necessary condition); then one table bit answers for all of them if the ring confirms that the neighbourhood is
                // one gray value.  A lane-divergent branch that textured content does not take.  (Testing for identical values
                // BEFORE building the mask makes flat content another 3 % faster and textured content 2.5 % slower: measured.)
                if (my == (1u << NPX) - 1u) {
                    uint32_t same = 0;
#pragma unroll
                    for (int j = 0; j < NP; j++) same |= (lo2u(F[j]) ^ lo2u(F[0])) | (hi2u(F[j]) ^ lo2u(F[0]));
                    if (same == 0u) {
                        dec = blur_flat_lane<NPX>(geo.ring_lane, (rowaddr[0] - geo.ring_lane) / kRowB, tab, xp.fix.flat_dec, r);
                        if (dec == 1u) dec = my;
                    }
                }
                if (my) {
                    // the general case: the reference's sequence for each pixel inside the band
                    if (dec == 2u) dec = blur_replay_lane<NPX>(my, rowaddr, tab, xp.fix);
                    if constexpr (STATS) {
                        if (p.slow_counter) atomicAdd(p.slow_counter, (unsigned long long)__popc(my));
                    }
                    if (dec) apply_dec<NPX, kFracBits>(F, dec);   // 256 + n + fraction -> 256 + (n - 1) + fraction
                }
            }
            __syncwarp();  // every lane is done with the ring before the next step overwrites its oldest slot
        }
#pragma unroll
        for (int j = 0; j < NP; j++) F[j] = pk2u(lo2u(F[j]) & kBiasMask, hi2u(F[j]) & kBiasMask);   // kBias + floor(S)
    } else {
        const float sc = __uint_as_float(0x7f000000u);  // 2^127: q*2^-149 -> q*2^-22 (a normal float)
        const u64 SC = pk2(sc, sc);
#pragma unroll
        for (int j = 0; j < NP; j++) F[j] = mul2(Q[j], SC);
    }

    // ---- 3. Sobel, vertical pass first: output row yo = yb-1 reads rows yb-2, yb-1, yb -------------
    // BORDER_REFLECT_101 in y: row -1 -> row 1 (first output row), row H -> row H-2 (last output row;
    // this step's input row is a dummy then).  Only the SPECIAL copy of the row body carries these
    // checks; the caller runs it for the first and last trips of a segment only.
    if constexpr (SPECIAL) {
        if (yb == 1) {
#pragma unroll
            for (int j = 0; j < NP; j++) st.F2[j] = F[j];
        }
        if (yb == H) {
#pragma unroll
            for (int j = 0; j < NP; j++) F[j] = st.F2[j];
        }
    }
    const u64 TWO = pk2(2.f, 2.f);
    u64 Vs[NP], Vd[NP];   // Vs = f(yb-2) + 2 f(yb-1) + f(yb),  Vd = f(yb) - f(yb-2)
#pragma unroll
    for (int j = 0; j < NP; j++) {
        Vs[j] = fma2(TWO, st.F1[j], add2(st.F2[j], F[j]));
        Vd[j] = sub2(F[j], st.F2[j]);
    }
    // horizontal pass, BORDER_REFLECT_101 in x: gx = Vs[x+1] - Vs[x-1],  gy = Vd[x-1] + 2 Vd[x] + Vd[x+1]
    float sl = __shfl_up_sync(FULL, hi2(Vs[NP - 1]), 1), sr = __shfl_down_sync(FULL, lo2(Vs[0]), 1);
    float dl = __shfl_up_sync(FULL, hi2(Vd[NP - 1]), 1), dr = __shfl_down_sync(FULL, lo2(Vd[0]), 1);
    if (geo.edge_warp) {
        sl = geo.e_left ? lo2(Vs[1]) : sl;             // x = -1 -> x = 1
        dl = geo.e_left ? lo2(Vd[1]) : dl;
        sr = geo.e_right ? hi2(Vs[NP - 2]) : sr;       // x = W  -> x = W-2
        dr = geo.e_right ? hi2(Vd[NP - 2]) : dr;
    }
    auto cs = [&](int m) -> float { return m == -1 ? sl : m == NPX ? sr : m < NP ? lo2(Vs[m]) : hi2(Vs[m - NP]); };
    auto cd = [&](int m) -> float { return m == -1 ? dl : m == NPX ? dr : m < NP ? lo2(Vd[m]) : hi2(Vd[m - NP]); };
    {
        // m * OS has the integer round-half-even(m) as its bit pattern (denormal result)
        const float os = __uint_as_float(BLUR ? 1u /* 2^-149 */ : 0x00400000u /* 2^-127 */);
        const u64 OS = pk2(os, os);
        uint32_t q[NPX];
#pragma unroll
        for (int j = 0; j < NP; j++) {
            u64 gx, dsum;   // gx = Vs[m+1] - Vs[m-1], dsum = Vd[m-1] + Vd[m+1] of the pair (j, j + NP)
            if (j - 1 >= 0 && j + 1 < NP) {
                gx = sub2(Vs[j + 1], Vs[j - 1]);
                dsum = add2(Vd[j - 1], Vd[j + 1]);
            } else {   // a tap crosses the lane boundary or the middle of the lane: scalar halves, no pair construction
                gx = pk2(__fsub_rn(cs(j + 1), cs(j - 1)), __fsub_rn(cs(j + NP + 1), cs(j + NP - 1)));
                dsum = pk2(__fadd_rn(cd(j - 1), cd(j + 1)), __fadd_rn(cd(j + NP - 1), cd(j + NP + 1)));
            }
            const u64 gy = fma2(TWO, Vd[j], dsum);
            const u64 m2 = fma2(gx, gx, mul2(gy, gy));
            const u64 m = mul2(pk2(sqrt_approx(lo2(m2)), sqrt_approx(hi2(m2))), OS);
            q[j] = lo2u(m);
            q[j + NP] = hi2u(m);
        }
        const uint32_t ok = (!SPECIAL || (r >= geo.r_store && r <= geo.r_last)) ? geo.store_lane : 0u;
        const uint32_t w0 = i2ip(q[1], q[0], i2ip(q[3], q[2], 0u));
        if constexpr (NPX == 8) {
            const uint32_t w1 = i2ip(q[5], q[4], i2ip(q[7], q[6], 0u));
            asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %3, 0;\n\t@p st.global.v2.u32 [%0], {%1, %2};\n\t}"
                         ::"l"(geo.dst), "r"(w0), "r"(w1), "r"(ok) : "memory");
        } else {
            asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p st.global.u32 [%0], %1;\n\t}"
                         ::"l"(geo.dst), "r"(w0), "r"(ok) : "memory");
        }
    }
#pragma unroll
    for (int j = 0; j < NP; j++) {
        st.F2[j] = st.F1[j];
        st.F1[j] = F[j];
    }
    geo.dst += W;
}

// The rows of one segment.  Head: the warm-up rows and the first storing row (it may be frame row 0), one row
// per trip with the SPECIAL copy of the row body and a run-time slot of the raw-row ring.  Main loop: NB rows per
// trip with the plain copy and compile-time slots.  Tail: the remaining rows (the last may be frame row H-1), SPECIAL
// again.  Only the main loop is hot, so only its copies of the row body need to stay in the instruction cache.
// NB = rows in flight in the raw-row ring = the unroll of the main loop: 3 with the blur stage; 6 without it, where a
// row is consumed twice as fast and load latency is the top stall.
template <int NPX, int CN, bool BGR, bool BLUR, int NB, bool STATS>
__device__ __forceinline__ void run_rows_x2(WarpX<NPX, CN> &st, const X2Params &xp, GeoX &geo, int r)
{
    constexpr uint32_t kRowB = 32 * NPX * 4;
    constexpr uint32_t kRawB = 32 * NPX * CN;   // bytes of one raw row of the warp's band
    const FusedParams &p = xp.f;
    // head: up to the first storing row -- and, with the blur stage, until the newest gray row sits in the last slot of a
    // half ring (slot 2 or 5), so that the main loop's trips write whole halves
#pragma unroll 1
    for (; (r <= geo.r_store || (BLUR && (geo.slot != 2u && geo.slot != 5u))) && r < geo.r_last; r++) {
        step_x2<NPX, CN, BGR, BLUR, true, STATS, -1, NB>(st, geo.raw_lane + geo.rs * kRawB, xp, geo, r);
        geo.rs = geo.rs == (uint32_t)NB - 1u ? 0u : geo.rs + 1u;
    }
    // the main loop runs while all rows of a trip store and the row they fetch (NB ahead) lies inside the band: step s
    // advances freely iff s + NB - 1 < in_row0 + in_rows - 1
    const int r_main_last = min(geo.r_last - 1, p.in_row0 + p.in_rows - 1 - NB);
    static_assert(!BLUR || NB == 3, "the half-ring addressing assumes three rows per trip");
    if constexpr (BLUR) {
        geo.ringA = geo.ring_lane + (geo.slot == 2u ? 3u * kRowB : 0u);
        geo.ringB = geo.ring_lane + (geo.slot == 2u ? 0u : 3u * kRowB);
    }
    // the raw-row slots of the NB steps of a trip (a trip returns to the slot it started from)
    uint32_t ra[NB];
    {
        uint32_t s = geo.rs;
#pragma unroll
        for (int k = 0; k < NB; k++) {
            ra[k] = geo.raw_lane + s * kRawB;
            s = s == (uint32_t)NB - 1u ? 0u : s + 1u;
        }
    }
    const int r_main0 = r;
#pragma unroll 1
    for (; r + NB - 1 <= r_main_last; r += NB) {
        if constexpr (BLUR) {
            step_x2<NPX, CN, BGR, BLUR, false, STATS, 0, NB>(st, ra[0], xp, geo, r);
            step_x2<NPX, CN, BGR, BLUR, false, STATS, 1, NB>(st, ra[1], xp, geo, r + 1);
            step_x2<NPX, CN, BGR, BLUR, false, STATS, 2, NB>(st, ra[2], xp, geo, r + 2);
            const uint32_t t = geo.ringA;   // the half just written becomes "last trip's"
            geo.ringA = geo.ringB;
            geo.ringB = t;
        } else {
#pragma unroll
            for (int k = 0; k < NB; k++) step_x2<NPX, CN, BGR, BLUR, false, STATS, 0, NB>(st, ra[k], xp, geo, r + k);
        }
    }
    // newest row: last slot of the half written last.  Only if a trip ran: a segment of one output row leaves the head at r_last
    // with the newest row in slot 1 (neither 2 nor 5), and no trip follows -- the tail must keep the head's slot.
    if constexpr (BLUR) {
        if (r != r_main0) geo.slot = (geo.ringB - geo.ring_lane) / kRowB + 2u;
    }
#pragma unroll 1
    for (; r <= geo.r_last; r++) {
        step_x2<NPX, CN, BGR, BLUR, true, STATS, -1, NB>(st, geo.raw_lane + geo.rs * kRawB, xp, geo, r);
        geo.rs = geo.rs == (uint32_t)NB - 1u ? 0u : geo.rs + 1u;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");   // (rows fetched past the segment's end)
}

template <int NPX, int CN, bool BGR, bool BLUR, bool STATS = false>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, NPX == 8 ? ((BLUR || CN == 1) ? kMinBlocks8 : kMinBlocks8NoBlur) : kMinBlocks4)
fused_x2_kernel(const __grid_constant__ X2Params xp)
{
    constexpr int HALO = BLUR ? 3 : 1;  // input rows above/below an output row
    constexpr int kRowW = 32 * NPX;     // words per ring row
    constexpr int kBand = 30 * NPX;
    constexpr int NW = NPX * CN / 4;
    constexpr int NB = BLUR ? 3 : 6;    // rows in flight in the raw-row ring (run_rows_x2)
    const FusedParams &p = xp.f;

    __shared__ __align__(16) uint32_t ring[BLUR ? kWarpsPerBlock * kRing * kRowW : 4];
    constexpr int kRawW = 32 * NPX * CN / 4;   // words of one raw row of a warp's band
    __shared__ __align__(16) uint32_t raw_ring[kWarpsPerBlock * NB * kRawW];
    // no block-level barrier: the warps are independent from the first instruction on

    GeoX geo;
    geo.lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    geo.ring_lane = (uint32_t)__cvta_generic_to_shared(ring + (BLUR ? warp * kRing * kRowW : 0)) + 16u * (uint32_t)geo.lane;
    geo.ringA = geo.ringB = geo.ring_lane;
    geo.slot = 1u;   // seven head rows later the newest row sits in slot 2
    // A block is kWarpsPerBlock adjacent bands of one row segment.  (One band x four consecutive segments per block -- the band,
    // and with it "does this warp touch an image border", block-uniform -- was measured in round 2: the loop bounds then depend
    // on the warp, ptxas guards every shuffle with BRA.DIV, 733 instead of 647 hot instructions per trip; one-warp blocks, where
    // everything is uniform: 449 us against 431 us.)
    int bid = blockIdx.x;
    const int bg = bid % p.n_band_groups; bid /= p.n_band_groups;
    const int seg = bid % p.n_segs;
    const int frame = bid / p.n_segs;
    const int band = bg * kWarpsPerBlock + warp;
    if (band >= p.n_bands) return;  // warp-uniform

    const int W = p.W;
    const int xw0 = band * kBand;
    const int x = xw0 - NPX + NPX * geo.lane;      // first of this lane's pixels
    const bool in_img = (x >= 0) && (x < W);       // W % NPX == 0: a lane is fully inside or fully outside
    const int lane_last = (W - xw0) / NPX;         // lane holding the last NPX pixels of the row (may be > 31)
    geo.e_left = (band == 0) && geo.lane == 1;
    geo.e_right = geo.lane == lane_last;
    geo.edge_warp = band == 0 || lane_last <= 31;
    if constexpr (BLUR) {
        // this lane's column table for the cold paths (read and written by its own lane only: no barrier)
        const int cmin = band == 0 ? NPX : 0, cmax = min(lane_last, 31) * NPX + NPX - 1;   // first / last band column inside the image (0 = pixel 0 of lane 0)
        const int rel_lo = cmin - NPX * geo.lane + 2, rel_hi = cmax - NPX * geo.lane + 2;   // the same in lane-relative columns
        const int *lut = NPX == 8 ? c_ring_rel8.v : c_ring_rel4.v;
        uint32_t *tab = &s_lane_tab[threadIdx.x * kLaneTabWords];
#pragma unroll 1
        for (int rel = 0; rel < NPX + 4; rel++) tab[rel] = (uint32_t)lut[min(max(min(max(rel, rel_lo), rel_hi), 0), NPX + 3)];   // (lanes outside the image: any valid entry)
        tab[kLaneTabWords - 1] = 0u;   // blur_flat_lane's history
    }
    geo.need = !in_img ? 0u : geo.lane == 0 ? 1u << (NPX - 1) : geo.lane == 31 ? 1u : (1u << NPX) - 1u;
    const int ys = p.out_row0 + seg * p.seg_rows;
    const int ye = min(ys + p.seg_rows, p.out_row0 + p.out_rows);
    geo.r_store = ys + HALO;
    geo.r_last = ye - 1 + HALO;
    geo.in_pitch = (uint32_t)W * CN;
    const uint8_t *in_base = p.in + (size_t)frame * p.in_frame_bytes;
    geo.store_lane = ((geo.lane >= 1) && (geo.lane <= 30) && in_img) ? 1u : 0u;

    WarpX<NPX, CN> st;
#pragma unroll
    for (int j = 0; j < NPX / 2; j++) {
        st.F1[j] = st.F2[j] = 0ull;
        st.a0[j] = st.a1[j] = st.a2[j] = st.a3[j] = 0ull;
    }

    // Rows are clamped to the rows the input band holds.  The host guarantees the band covers every
    // row an output needs, and that it starts at row 0 / ends at row H-1 wherever the clamp-to-edge rule
    // (GaussianBlur.cpp:241) is actually exercised; other clamped rows are read-ahead only.
    int r = ys - HALO;
    const uint32_t xoff = in_img ? (uint32_t)x * CN : 0u;
    geo.raw_lane = (uint32_t)__cvta_generic_to_shared(raw_ring + warp * NB * kRawW) + (uint32_t)(NPX * CN) * (uint32_t)geo.lane;
    geo.rs = 0u;
#pragma unroll
    for (int k = 0; k < NB; k++) {   // rows r .. r + NB - 1 into slots 0 .. NB - 1
        const int i = min(max(r + k - p.in_row0, 0), p.in_rows - 1);
        geo.src = in_base + (size_t)i * geo.in_pitch + xoff;
        cp_row_x3<NPX, CN>(geo.raw_lane + (uint32_t)k * (uint32_t)(kRawW * 4), geo.src);
    }
    // step r fetches row r + NB = one past the row src points at: advance iff in_row0 <= r + NB - 1 < in_row0 + in_rows - 1
    geo.adv_lo = p.in_row0 - (NB - 1);
    geo.adv_n = p.in_rows - 1;
    // output row produced by the step of input row r is r - HALO
    geo.dst = p.out + (size_t)frame * p.out_rows * W + (ptrdiff_t)(r - HALO - p.out_row0) * W + x;

    run_rows_x2<NPX, CN, BGR, BLUR, NB, STATS>(st, xp, geo, r);
}
