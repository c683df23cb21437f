// ofdm_device.cuh -- device-side building blocks of the B200 802.11a OFDM stage chain.
//
// Work decomposition (all kernels): a warp is four 8-lane groups; each group owns one
// 64-point FFT window (an LTS half or one OFDM symbol body) held in registers, 8 complex
// values per lane.  Lane u of a group owns time samples {u + 8m} on the way in and FFT bins
// {u + 8j} on the way out, so global loads/stores are 64-byte contiguous per group and the
// only cross-lane traffic inside a transform is one 8x8 transpose through a padded,
// bank-conflict-free shared-memory tile.
//
// Two arithmetic modes share the layout:
//   EXACT  bit-for-bit the reference's recursive radix-2 DIT (src/OFDM.c:282-312): six
//          butterfly stages, twiddle products in double (no FMA contraction) rounded to float,
//          float add/sub.  The dataflow, not the schedule, defines the bits (SURVEY.md sec. 7).
//   FAST   fp32 8x8 Cooley-Tukey (radix-8 in registers, float twiddles, FMA).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "twiddles64.h"

namespace ofdm {

constexpr int kGroupPitch = 72;          // float2 per 8-lane transpose tile (8 rows x 9)
constexpr int kWarpTile = 4 * kGroupPitch;
constexpr float kQpsk = 0.70710678118654752440f;   // (float)(1/sqrt(2)) = 0x3F3504F3, OFDM.c:424

// W_64^k in double exactly as the reference evaluates cexp(-I*2.0*PI*k/sz) (generated header)
constexpr double kTw64[32][2] = { OFDM_TWIDDLE64_TABLE };
// the three lane-independent twiddles of the in-lane stages, as scalars usable in device code
constexpr double kW8r = kTw64[8][0],   kW8i = kTw64[8][1];      // W_8^1
constexpr double kW16r = kTw64[16][0], kW16i = kTw64[16][1];    // W_4^1 = W_8^2 (6.1e-17, -1): NOT special-cased
constexpr double kW24r = kTw64[24][0], kW24i = kTw64[24][1];    // W_8^3
constexpr double kW8rS = kTw64[8][0] * 0x1p896, kW8iS = kTw64[8][1] * 0x1p896;       // the same, pre-scaled for bf_exact_s
constexpr double kW24rS = kTw64[24][0] * 0x1p896, kW24iS = kTw64[24][1] * 0x1p896;

struct Tables {
    double2 tw64[32];       // exact twiddles
    float2 tw64f[64];       // fp32 twiddles W_64^k, k = 0..63
    int8_t bin_data[64];    // natural bin p -> data index 0..47, -1 null, -2 pilot +1, -3 pilot -1
    int8_t bin_lts[64];     // natural bin p -> L value (+1, -1, 0)   OFDM.c:494
    int8_t data_bin[48];    // data index -> natural bin p (inverse of bin_data)
    float2 lts_time[160];   // LTS slot in time (filled by the exact ifft at context creation)
    float lts_power_prefix; // exact-mode running float power sum after the 160 LTS samples (OFDM.c:637-641)
    float lts_power_sum;    // sum |lts|^2 over the 160 LTS samples (fast mode)
};
__constant__ Tables c_tab;

__device__ __forceinline__ int rev3(int v) { return ((v & 1) << 2) | (v & 2) | ((v >> 2) & 1); }

// ---------------------------------------------------------------- packed fp32 (sm_100 FADD2 / FMUL2 / FFMA2)
// A complex value is a float2 = one 64-bit register pair, and Blackwell's packed fp32 instructions operate on such
// pairs lane by lane with round-to-nearest per lane: one issue slot per complex add instead of two.  Their operands
// take a swap (LO_HI), per-lane negation and a scalar broadcast for free, so a rotation by -i, a conjugate or
// "real part times complex" cost nothing extra: ptxas folds the make_float2() shuffles below into operand modifiers
// (profiles/r2_sass_*.txt: no MOV / PRMT around them).  Every helper is bit-identical to the scalar expression in
// its comment.
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ float2 cadd_mi(float2 a, float2 b) { return __fadd2_rn(a, make_float2(b.y, -b.x)); }   // a + b*(-i)
__device__ __forceinline__ float2 csub_mi(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.y, b.x)); }   // a - b*(-i)
// (fma(a.x, b.x, -(a.y*b.y)), fma(a.x, b.y, a.y*b.x)): FMUL2 with a broadcast, FFMA2 with a mixed-sign addend
__device__ __forceinline__ float2 cmul(float2 a, float2 b)
{
    const float2 t = __fmul2_rn(make_float2(a.y, a.y), make_float2(b.y, b.x));
    return __ffma2_rn(make_float2(a.x, a.x), b, make_float2(-t.x, t.y));
}

// ---------------------------------------------------------------- exact-mode butterflies
// W * o with W double, o float promoted: (wr*c - wi*d) + i(wr*d + wi*c), each op rounded
// separately (gcc without -mfma), then rounded to float; e +- that in float.  OFDM.c:303-305
__device__ __forceinline__ void bf_exact(float2 &e, float2 &o, double wr, double wi)
{
    double c = (double)o.x, d = (double)o.y;
    const float2 w = make_float2(__double2float_rn(__dsub_rn(__dmul_rn(wr, c), __dmul_rn(wi, d))),
                                 __double2float_rn(__dadd_rn(__dmul_rn(wr, d), __dmul_rn(wi, c))));
    const float2 a = e;
    e = cadd(a, w); o = csub(a, w);
}
// float -> double without the XU pipe.  The float's bits are re-laid as a double with the SAME biased exponent
// field, i.e. the value x * 2^-896 (exact for normals, denormals and zeros: a zero exponent field means
// 0.m * 2^-1022 there and 0.m * 2^-126 here).  The missing 2^896 is folded into the twiddle, so the double product
// W * x has the same real value and therefore the same rounding as the reference's.  (Non-finite samples are not
// reproduced by this path.)
constexpr double kTwScale = 0x1p896;
__device__ __forceinline__ double f2d_scaled(float x)
{
    const uint32_t u = __float_as_uint(x);
    const uint32_t hi = ((u << 1) >> 4) | (u & 0x80000000u);
    return __hiloint2double((int)hi, (int)(u << 29));
}
// same butterfly as bf_exact with pre-scaled twiddles (wr, wi already multiplied by 2^896)
__device__ __forceinline__ void bf_exact_s(float2 &e, float2 &o, double wr, double wi)
{
    const double c = f2d_scaled(o.x), d = f2d_scaled(o.y);
    const float2 w = make_float2(__double2float_rn(__dsub_rn(__dmul_rn(wr, c), __dmul_rn(wi, d))),
                                 __double2float_rn(__dadd_rn(__dmul_rn(wr, d), __dmul_rn(wi, c))));
    const float2 a = e;
    e = cadd(a, w); o = csub(a, w);
}
// k = 0: W = (1, -0); the product equals o for every finite o (up to the sign of a zero)
__device__ __forceinline__ void bf_unit(float2 &e, float2 &o)
{
    const float2 a = e, w = o;
    e = cadd(a, w); o = csub(a, w);
}

// k = sz/4: W = (6.1e-17, -1) exactly as cexp() returns it.  The product is
// (fl64(wr*c) + d, fl64(wr*d) - c) rounded to float, which is (d, -c) unless the 2^-53.9-scaled
// term reaches a quarter ulp of the float it is added to (|c| >= 1.2e8 |d|, or d == 0): those
// inputs (exact zeros in noise-free frames, mostly) take the full double product.
__device__ __forceinline__ void bf_quarter(float2 &e, float2 &o)
{
    const float c = o.x, d = o.y;
    if (fabsf(c) * 1e-8f < fabsf(d) && fabsf(d) * 1e-8f < fabsf(c)) {
        const float2 a = e, w = o;
        e = cadd_mi(a, w); o = csub_mi(a, w);           // a +- (d, -c)
    } else {
        bf_exact(e, o, kW16r, kW16i);
    }
}

struct TwExact { double2 w16, w32a, w32b, w64a, w64b, w64c, w64d; };

__device__ __forceinline__ TwExact load_tw_exact(int t)
{
    TwExact w;
    w.w16 = c_tab.tw64[4 * t];
    w.w32a = c_tab.tw64[2 * t];  w.w32b = c_tab.tw64[2 * t + 16];
    w.w64a = c_tab.tw64[t];      w.w64b = c_tab.tw64[t + 8];
    w.w64c = c_tab.tw64[t + 16]; w.w64d = c_tab.tw64[t + 24];
    // pre-scaled by 2^896 for bf_exact_s (exact: a power of two, no overflow for |w| <= 1)
    // The exact butterflies are bound by the XU pipe (F2F) on one side and by instruction issue on the other: widening
    // on the ALU costs four instructions instead of one.  Measured optimum on B200: stages 32 and 64 widen on the ALU
    // (their twiddles carry the 2^896), the in-lane stages and stage 16 keep F2F.
    double2 *all[6] = {&w.w32a, &w.w32b, &w.w64a, &w.w64b, &w.w64c, &w.w64d};
#pragma unroll
    for (int i = 0; i < 6; ++i) { all[i]->x = __dmul_rn(all[i]->x, kTwScale); all[i]->y = __dmul_rn(all[i]->y, kTwScale); }
    return w;
}

// in : v[i] = x[8*rev3(i) + u]  (bit-reversed placement: lane u, slot i is position 8*rev3(u)+i)
// out: v[j] = X[u + 8j]         (natural bins, not yet fft_shift'ed)
__device__ __forceinline__ void fft64_exact(float2 (&v)[8], const TwExact &tw, float2 *tile, int u)
{
    // sz = 2, 4, 8 inside the lane (positions 8t..8t+7)
    bf_unit(v[0], v[1]); bf_unit(v[2], v[3]); bf_unit(v[4], v[5]); bf_unit(v[6], v[7]);
    bf_unit(v[0], v[2]); bf_quarter(v[1], v[3]);
    bf_unit(v[4], v[6]); bf_quarter(v[5], v[7]);
    bf_unit(v[0], v[4]);
    bf_exact(v[1], v[5], kW8r, kW8i);              // the in-lane stages keep the XU conversion: the two pipes share the load
    bf_quarter(v[2], v[6]);
    bf_exact(v[3], v[7], kW24r, kW24i);
    // 8x8 transpose: position q = 8*rev3(u) + i  ->  lane q%8, slot q/8
    const int row = rev3(u) * 9;
#pragma unroll
    for (int i = 0; i < 8; ++i) tile[row + i] = v[i];
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = tile[j * 9 + u];
    __syncwarp();
    // sz = 16, 32, 64 on positions u + 8j
    bf_exact(v[0], v[1], tw.w16.x, tw.w16.y); bf_exact(v[2], v[3], tw.w16.x, tw.w16.y);
    bf_exact(v[4], v[5], tw.w16.x, tw.w16.y); bf_exact(v[6], v[7], tw.w16.x, tw.w16.y);
    bf_exact_s(v[0], v[2], tw.w32a.x, tw.w32a.y); bf_exact_s(v[1], v[3], tw.w32b.x, tw.w32b.y);
    bf_exact_s(v[4], v[6], tw.w32a.x, tw.w32a.y); bf_exact_s(v[5], v[7], tw.w32b.x, tw.w32b.y);
    bf_exact_s(v[0], v[4], tw.w64a.x, tw.w64a.y); bf_exact_s(v[1], v[5], tw.w64b.x, tw.w64b.y);
    bf_exact_s(v[2], v[6], tw.w64c.x, tw.w64c.y); bf_exact_s(v[3], v[7], tw.w64d.x, tw.w64d.y);
}

// ---------------------------------------------------------------- fast-mode fp32 transform
// forward 8-point DFT, natural order in and out (decimation in frequency); 28 packed instructions
__device__ __forceinline__ void dft8(float2 (&v)[8])
{
    const float h = 0.70710678118654752440f;
    const float2 hh = make_float2(h, h);
    const float2 a0 = cadd(v[0], v[4]), b0 = csub(v[0], v[4]);
    const float2 a1 = cadd(v[1], v[5]), b1d = csub(v[1], v[5]);
    const float2 a2 = cadd(v[2], v[6]), b2 = csub(v[2], v[6]);          // b2 * W8^2 = b2 * (-i): folded into its consumers
    const float2 a3 = cadd(v[3], v[7]), b3d = csub(v[3], v[7]);
    const float2 b1 = __fmul2_rn(cadd_mi(b1d, b1d), hh);                                                         // * W8^1: ((x+y)h, (y-x)h)
    const float2 b3 = __fmul2_rn(__fadd2_rn(make_float2(b3d.y, -b3d.x), make_float2(-b3d.x, -b3d.y)), hh);       // * W8^3: ((y-x)h, -(x+y)h)
    const float2 s0 = cadd(a0, a2), s1 = csub(a0, a2), s2 = cadd(a1, a3), d3 = csub(a1, a3);
    v[0] = cadd(s0, s2); v[4] = csub(s0, s2); v[2] = cadd_mi(s1, d3); v[6] = csub_mi(s1, d3);
    const float2 t0 = cadd_mi(b0, b2), t1 = csub_mi(b0, b2), t2 = cadd(b1, b3), e3 = csub(b1, b3);
    v[1] = cadd(t0, t2); v[5] = csub(t0, t2); v[3] = cadd_mi(t1, e3); v[7] = csub_mi(t1, e3);
}

struct TwFast { float2 w[7]; };    // W_64^(u*k), k = 1..7

__device__ __forceinline__ TwFast load_tw_fast(int u)
{
    TwFast t;
#pragma unroll
    for (int k = 1; k < 8; ++k) t.w[k - 1] = c_tab.tw64f[u * k];
    return t;
}

// in : v[m] = x[u + 8m];  out: v[j] = X[u + 8j]
__device__ __forceinline__ void fft64_fast(float2 (&v)[8], const TwFast &tw, float2 *tile, int u)
{
    dft8(v);
#pragma unroll
    for (int k = 1; k < 8; ++k) v[k] = cmul(v[k], tw.w[k - 1]);
    const int row = u * 9;
#pragma unroll
    for (int k = 0; k < 8; ++k) tile[row + k] = v[k];
    __syncwarp();
#pragma unroll
    for (int m = 0; m < 8; ++m) v[m] = tile[m * 9 + u];
    __syncwarp();
    dft8(v);
}

template <bool EXACT> struct Tw;
template <> struct Tw<true>  { TwExact t; __device__ __forceinline__ void load(int u) { t = load_tw_exact(u); } };
template <> struct Tw<false> { TwFast t;  __device__ __forceinline__ void load(int u) { t = load_tw_fast(u); } };

// slot -> which multiple of 8 the lane's input sample sits at
template <bool EXACT> __device__ __forceinline__ int slot_m(int i) { return EXACT ? rev3(i) : i; }

template <bool EXACT>
__device__ __forceinline__ void fft64(float2 (&v)[8], const Tw<EXACT> &tw, float2 *tile, int u)
{
    if constexpr (EXACT) fft64_exact(v, tw.t, tile, u); else fft64_fast(v, tw.t, tile, u);
}

// ---------------------------------------------------------------- bits / constellation
// data index d of a symbol -> its two payload bits (a = bit 2d, b = bit 2d+1)
__device__ __forceinline__ uint32_t bit_pair(uint32_t w0, uint32_t w1, uint32_t w2, int d)
{
    uint32_t w = d < 16 ? w0 : (d < 32 ? w1 : w2);
    return (w >> (2 * (d & 15))) & 3u;          // bit0 = a, bit1 = b
}
// QPSK_Modulator OFDM.c:423-430: 00->(+,+) 01->(-,+) 10->(-,-) 11->(+,-)
__device__ __forceinline__ float2 qpsk_point(uint32_t ab)
{
    uint32_t a = ab & 1u, b = ab >> 1;
    return make_float2((a ^ b) ? -kQpsk : kQpsk, a ? -kQpsk : kQpsk);
}
// AGC_Receiver :860-868 followed by QPSK_Demodulator :883-902 on the rail signs
__device__ __forceinline__ uint32_t demod_pair(bool re_pos, bool im_pos)
{
    uint32_t a = im_pos ? 0u : 1u, b = (re_pos != im_pos) ? 1u : 0u;
    return a | (b << 1);
}

// ---------------------------------------------------------------- glibc-faithful hypot (exact P)
// cabs() of the promoted sample in Transmission_Over_Air (OFDM.c:640) is glibc 2.39 hypot(), whose
// non-FMA kernel (sqrt + one correction step) is made of IEEE basic operations only; reproduced
// with round-to-nearest intrinsics.  Inputs here are float-valued, so no scaling branch is needed
// except the "ay negligible" shortcut.
__device__ __forceinline__ double hypot_glibc(double x, double y)
{
    x = fabs(x); y = fabs(y);
    double ax = x < y ? y : x, ay = x < y ? x : y;
    if (ax >= __dmul_rn(ay, 0x1p54)) return __dadd_rn(ax, ay);      // ay / EPS, EPS = 2^-54: exact scaling
    double h = __dsqrt_rn(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)));
    double t1, t2;
    if (h <= __dmul_rn(2.0, ay)) {
        double delta = __dsub_rn(h, ay);
        t1 = __dmul_rn(ax, __dsub_rn(__dmul_rn(2.0, delta), ax));
        t2 = __dmul_rn(__dsub_rn(delta, __dmul_rn(2.0, __dsub_rn(ax, ay))), delta);
    } else {
        double delta = __dsub_rn(h, ax);
        t1 = __dmul_rn(__dmul_rn(2.0, delta), __dsub_rn(ax, __dmul_rn(2.0, ay)));
        t2 = __dadd_rn(__dmul_rn(__dsub_rn(__dmul_rn(4.0, delta), ay), ay), __dmul_rn(delta, delta));
    }
    return __dsub_rn(h, __ddiv_rn(__dadd_rn(t1, t2), __dmul_rn(2.0, h)));
}

// ---------------------------------------------------------------- Philox4x32-10 + Box-Muller
struct Philox {
    static constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
    __device__ __forceinline__ static uint4 run(uint4 c, uint32_t k0, uint32_t k1)
    {
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            uint32_t h0 = __umulhi(M0, c.x), l0 = M0 * c.x;
            uint32_t h1 = __umulhi(M1, c.z), l1 = M1 * c.z;
            c = make_uint4(h1 ^ c.y ^ k0, l1, h0 ^ c.w ^ k1, l0);
            k0 += W0; k1 += W1;
        }
        return c;
    }
};
// domain 3 is the flat noise layout of k_awgn_philox_flat; domain 4 holds the Q-rail draws of complex noise, in the block
// layout of domain 0 (noise_slot), so that a complex channel's I-rail draws are exactly those of the real-rail channel
enum { kDomainNoise = 0, kDomainBits = 1, kDomainTaps = 2, kDomainNoiseQ = 4 };

// one Box-Muller pair from two words (both branches used); fast intrinsics
__device__ __forceinline__ float2 box_muller(uint32_t r0, uint32_t r1)
{
    float u1 = fmaf((float)r0, 0x1p-32f, 0x1p-33f);
    float u2 = (float)r1 * 0x1p-32f;
    float rad;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad) : "f"(-2.0f * __logf(u1)));
    float s, c;
    __sincosf(6.283185307179586f * u2, &s, &c);
    return make_float2(rad * c, rad * s);
}
__device__ __forceinline__ void philox_normals4(uint32_t seed, uint32_t stream, uint64_t frame, uint32_t blk,
                                                uint32_t domain, float (&z)[4])
{
    uint4 r = Philox::run(make_uint4((uint32_t)frame, (uint32_t)(frame >> 32), blk, domain), seed, stream);
    float2 p = box_muller(r.x, r.y), q = box_muller(r.z, r.w);
    z[0] = p.x; z[1] = p.y; z[2] = q.x; z[3] = q.y;
}
// first Philox block of the 64-sample window that starts at frame sample n0 (see DESIGN.md
// "Philox streams"; mirrored by noise_slot() in oracle/ofdm_oracle.c)
__device__ __forceinline__ int window_block_base(int n0)
{
    if (n0 < 160) return n0 < 96 ? 8 : 24;
    int s = (n0 - 176) / 80;
    return 44 + 20 * s;
}

// ---------------------------------------------------------------- reductions
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ uint32_t warp_sum(uint32_t v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace ofdm
