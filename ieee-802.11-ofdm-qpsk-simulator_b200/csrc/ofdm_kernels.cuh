// ofdm_kernels.cuh -- the __global__ kernels of the stage chain (see ofdm_device.cuh for the
// work decomposition).  Included once, by ofdm_b200.cu.
#pragma once
#include "ofdm_device.cuh"
#include "../../include/ofdm_b200.h"

namespace ofdm {

constexpr int kWarpsPerBlock = 8;
constexpr int kThreads = kWarpsPerBlock * 32;
enum { kNoiseNone = 0, kNoiseInject = 1, kNoisePhilox = 2 };

// ------------------------------------------------------------------ layout helpers
// one byte per bit -> 3 packed words per symbol (OFDM.c stores bits as float complex; the
// byte form is what a host-side caller naturally has)
__global__ void k_pack_bits(const uint8_t *__restrict__ bits, uint32_t *__restrict__ packed, long n_words)
{
    long w = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_words) return;
    const uint8_t *b = bits + w * 32;
    uint32_t v = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) v |= (uint32_t)(b[j] & 1u) << j;
    packed[w] = v;
}
__global__ void k_unpack_bits(const uint32_t *__restrict__ packed, uint8_t *__restrict__ bits, long n_bits)
{
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_bits) return;
    bits[i] = (uint8_t)((packed[i >> 5] >> (i & 31)) & 1u);
}

// The element-wise stages below share one shape: a block covers four rows (symbols) per step of a grid-stride loop and a
// thread keeps its column for the whole launch, so everything that depends only on the column -- which payload word and
// bit pair, which source bin, which table entry (a lane-varying index into __constant__ memory is read once per thread,
// not once per element) -- is computed once, nothing divides per element, and every row is read and written as one
// contiguous run.  Block sizes: 4 x columns (kRows4).
constexpr int kRows4 = 4;

// QPSK_Modulator OFDM.c:415-433; column = constellation point d of the symbol (block of 4 x 48 threads)
__global__ void __launch_bounds__(kRows4 * 48) k_qpsk_mod(const uint32_t *__restrict__ bits, float2 *__restrict__ mod, long n_sym_total)
{
    const int d = threadIdx.x % 48, r = threadIdx.x / 48;
    const int word = d >> 4, shift = 2 * (d & 15);
    for (long sym = (long)blockIdx.x * kRows4 + r; sym < n_sym_total; sym += (long)gridDim.x * kRows4)
        mod[sym * 48 + d] = qpsk_point((bits[sym * 3 + word] >> shift) & 3u);
}
// the same on a 16-byte aligned output: two points per store (block of 4 x 24 threads x 2 row groups)
__global__ void __launch_bounds__(2 * kRows4 * 24) k_qpsk_mod2(const uint32_t *__restrict__ bits, float4 *__restrict__ mod, long n_sym_total)
{
    const int h = threadIdx.x % 24, r = threadIdx.x / 24;           // points 2h, 2h + 1 of the symbol
    const int word = h >> 3, shift = 4 * (h & 7);
    for (long sym = (long)blockIdx.x * (2 * kRows4) + r; sym < n_sym_total; sym += (long)gridDim.x * (2 * kRows4)) {
        const uint32_t q = bits[sym * 3 + word] >> shift;
        const float2 a = qpsk_point(q & 3u), b = qpsk_point((q >> 2) & 3u);
        mod[sym * 24 + h] = make_float4(a.x, a.y, b.x, b.y);
    }
}

// frame-build block OFDM.c:523-548; column = grid bin (centred index c) (block of 4 x 64 threads)
__global__ void __launch_bounds__(kRows4 * 64) k_map_subcarriers(const float2 *__restrict__ mod, float2 *__restrict__ grid, long n_sym_total)
{
    const int c = threadIdx.x & 63, r = threadIdx.x >> 6;
    const int d = c_tab.bin_data[(c + 32) & 63];
    const float2 fixed = make_float2(d == -2 ? 1.f : (d == -3 ? -1.f : 0.f), 0.f);            // pilots {1,1,1,-1} :523, nulls
    for (long sym = (long)blockIdx.x * kRows4 + r; sym < n_sym_total; sym += (long)gridDim.x * kRows4)
        grid[sym * 64 + c] = d >= 0 ? mod[sym * 48 + d] : fixed;
}

// CP add OFDM.c:559-565; column = output sample k of the 80 (block of 4 x 80 threads)
__global__ void __launch_bounds__(kRows4 * 80) k_add_cp(const float2 *__restrict__ sym, float2 *__restrict__ out, long n_sym_total)
{
    const int k = threadIdx.x % 80, r = threadIdx.x / 80;
    const int src = k < 16 ? 48 + k : k - 16;
    for (long s = (long)blockIdx.x * kRows4 + r; s < n_sym_total; s += (long)gridDim.x * kRows4)
        out[s * 80 + k] = sym[s * 64 + src];
}

// ------------------------------------------------------------------ stand-alone transforms
// fft OFDM.c:314-318 (INVERSE = false) and ifft OFDM.c:320-339 (INVERSE = true) on [n][64]
// centred buffers, one 8-lane group per transform.
template <bool EXACT, bool INVERSE>
__global__ void __launch_bounds__(kThreads) k_fft64(const float2 *__restrict__ in, float2 *__restrict__ out, long n)
{
    __shared__ float2 s_tile[kWarpsPerBlock][kWarpTile];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, u = lane & 7;
    float2 *tile = s_tile[warp] + grp * kGroupPitch;
    Tw<EXACT> tw; tw.load(u);
    const long n_groups = (long)gridDim.x * kWarpsPerBlock * 4;
    const long iters = (n + n_groups - 1) / n_groups;
    for (long it = 0; it < iters; ++it) {
        long t = it * n_groups + ((long)blockIdx.x * kWarpsPerBlock + warp) * 4 + grp;
        bool active = t < n;
        float2 v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int nn = 8 * slot_m<EXACT>(i) + u;                 // natural input index
            float2 x = make_float2(0.f, 0.f);
            if (active) {
                if (INVERSE) { x = in[t * 64 + ((nn + 32) & 63)]; x.y = -x.y; }   // ifft_shift :208 + conj :328
                else x = in[t * 64 + nn];
            }
            v[i] = x;
        }
        fft64<EXACT>(v, tw, tile, u);
        if (active) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                int c = (u + 8 * j + 32) & 63;                  // fft_shift :227
                float2 y = v[j];
                if (INVERSE) { y.x = y.x * 0.015625f; y.y = -y.y * 0.015625f; }   // conj, /sz :334 (exact scaling)
                out[t * 64 + c] = y;
            }
        }
    }
}

// ------------------------------------------------------------------ transmitter
// Transmitter OFDM.c:500-581 (QPSK map, subcarrier/pilot map, ifft, CP, LTS || data concat) fused:
// bits in, frame IQ out, nothing else touches HBM.  One 8-lane group per OFDM symbol.
template <bool EXACT>
__global__ void __launch_bounds__(kThreads) k_tx_frames(const uint32_t *__restrict__ bits, float2 *__restrict__ frames,
                                                        long n_frames, int n_sym)
{
    __shared__ float2 s_tile[kWarpsPerBlock][kWarpTile];
    __shared__ __align__(16) float2 s_lts_time[160];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, u = lane & 7;
    float2 *tile = s_tile[warp] + grp * kGroupPitch;
    Tw<EXACT> tw; tw.load(u);
    int dmap[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) dmap[i] = c_tab.bin_data[8 * slot_m<EXACT>(i) + u];   // input index n <-> centred (n+32)%64
    for (int i = threadIdx.x; i < 160; i += kThreads) s_lts_time[i] = c_tab.lts_time[i];
    __syncthreads();
    const int len = 160 + 80 * n_sym;
    const long n_symbols = n_frames * n_sym;
    const long n_groups = (long)gridDim.x * kWarpsPerBlock * 4;
    const long iters = (n_symbols + n_groups - 1) / n_groups;
    for (long it = 0; it < iters; ++it) {
        long t = it * n_groups + ((long)blockIdx.x * kWarpsPerBlock + warp) * 4 + grp;
        bool active = t < n_symbols;
        uint32_t w0 = 0, w1 = 0, w2 = 0;
        if (active) { const uint32_t *w = bits + t * 3; w0 = w[0]; w1 = w[1]; w2 = w[2]; }
        float2 v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            // grid value at centred index (n+32)%64 (ifft_shift :208), conjugated (:328)
            int d = dmap[i];
            float2 x = make_float2(0.f, -0.f);
            if (d >= 0) { x = qpsk_point(bit_pair(w0, w1, w2, d)); x.y = -x.y; }
            else if (d == -2) x.x = 1.f;
            else if (d == -3) x.x = -1.f;
            v[i] = x;
        }
        fft64<EXACT>(v, tw, tile, u);
        if (active) {
            long f = t / n_sym; int s = (int)(t - f * n_sym);
            float2 *fr = frames + f * len;
            float2 *dst = fr + 160 + 80 * s;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                int np = u + 8 * ((j + 4) & 7);                 // fft_shift inside ifft's fft() -> 32-sample rotation (Q4)
                float2 y = make_float2(v[j].x * 0.015625f, -v[j].y * 0.015625f);
                dst[16 + np] = y;                               // body :564
                if (np >= 48) dst[np - 48] = y;                 // CP   :563
            }
            if (s == 0) {                                       // LTS slot :573 (constant, built at context creation)
                const float4 *src4 = reinterpret_cast<const float4 *>(s_lts_time);
                float4 *dst4 = reinterpret_cast<float4 *>(fr);              // frames are 2560 B: 16-byte aligned
#pragma unroll
                for (int k = 0; k < 10; ++k) dst4[u + 8 * k] = src4[u + 8 * k];
            }
        }
    }
}

// signal power of Transmission_Over_Air OFDM.c:637-643.  EXACT: double terms cabs*cabs (glibc hypot), accumulated
// sequentially into a float.  The chain is inherently serial per frame, so every lane runs the chain of its own
// frame (32 frames per warp in flight); a lane walks its frame 16 bytes at a time, so each 128-byte line it
// touches is fetched once and served from L1 for the next seven loads.  `first` / `acc0` let the transmitter
// skip the LTS slot, whose partial sum is a constant of the build (Tables::lts_power_prefix).
template <bool VEC>
__global__ void __launch_bounds__(kThreads) k_frame_power_exact(const float2 *__restrict__ frames, float *__restrict__ power,
                                                                long n_frames, int len, int first, float acc0)
{
    const long f = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames) return;
    float p = acc0;
    if (VEC) {
        const float4 *x = reinterpret_cast<const float4 *>(frames + f * len + first);     // first and len are even, base 16-byte aligned
        const int n2 = (len - first) >> 1;
#pragma unroll 2
        for (int i = 0; i < n2; ++i) {
            const float4 s = x[i];
            const double h0 = hypot_glibc((double)s.x, (double)s.y);
            const double h1 = hypot_glibc((double)s.z, (double)s.w);
            p = __double2float_rn(__dadd_rn((double)p, __dmul_rn(h0, h0)));
            p = __double2float_rn(__dadd_rn((double)p, __dmul_rn(h1, h1)));
        }
    } else {
        const float2 *x = frames + f * len;
        for (int i = 0; i < len; ++i) {
            const float2 s = x[i];
            const double h = hypot_glibc((double)s.x, (double)s.y);
            p = __double2float_rn(__dadd_rn((double)p, __dmul_rn(h, h)));
        }
    }
    power[f] = __fdiv_rn(p, (float)len);
}
// The same chain at memory speed (frames whose summed part is a whole number of 16-sample chunks, i.e. every transmitter
// frame).  Two changes against k_frame_power_exact, neither visible in the result:
//  * a warp fetches 32 frames x one 128-byte chunk with coalesced 16-byte loads (four rows per instruction) and turns the
//    tile through shared memory (row pitch 144 bytes: conflict-free both ways), so every line crosses the chip once and
//    nothing depends on 2048 threads' lines surviving in L1;
//  * the term of a sample is speculated as t = fma(x, x, y*y) in double instead of hypot()^2.  glibc's hypot is within one
//    ulp of sqrt(x^2 + y^2), so its rounded square is within 5 ulps of x^2 + y^2 and t within 1: the two double sums p + term
//    differ by at most 7 ulps.  They round to the same float unless the speculated sum lies within `margin` (16) double ulps
//    of a tie between two floats (its low 29 bits next to 2^28) -- 6e-8 of the samples, which take the reference's
//    operations instead.  The accumulator stays a float-valued double: away from a tie, rounding to float is adding 2^28
//    to the low word and clearing 29 bits.  Sums outside [1e-30, 1e30] (float subnormals, overflow, NaN) are never speculated.
//    margin = 2^28 sends every sample through the reference's operations (tests compare the two bit for bit).
__device__ __forceinline__ double power_step(double pd, float x, float y, uint32_t margin)
{
    const double dx = (double)x, dy = (double)y;
    const double s = __dadd_rn(pd, __fma_rn(dx, dx, __dmul_rn(dy, dy)));
    const uint32_t lo = (uint32_t)__double2loint(s), hi = (uint32_t)__double2hiint(s);
    const int dist = (int)(lo & 0x1fffffffu) - 0x10000000;
    const bool ok = (uint32_t)(dist < 0 ? -dist : dist) > margin && s > 1e-30 && s < 1e30;
    if (!ok) {                                                      // the reference's operations, OFDM.c:640-641
        const double h = hypot_glibc(dx, dy);
        return (double)__double2float_rn(__dadd_rn(pd, __dmul_rn(h, h)));
    }
    const uint32_t lo2 = lo + 0x10000000u;
    return __hiloint2double((int)(hi + (lo2 < lo ? 1u : 0u)), (int)(lo2 & 0xe0000000u));
}
constexpr int kPowPitch = 9;                                        // float4 per tile row: 8 data + 1 pad
__global__ void __launch_bounds__(kThreads) k_frame_power_tiled(const float2 *__restrict__ frames, float *__restrict__ power,
                                                                long n_frames, int len, int first, float acc0, uint32_t margin)
{
    __shared__ float4 s_tile[kWarpsPerBlock][32 * kPowPitch];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long f0 = ((long)blockIdx.x * kWarpsPerBlock + warp) * 32;
    if (f0 >= n_frames) return;
    float4 *tile = s_tile[warp];
    const int col = lane & 7, r0 = lane >> 3;
    const int n_chunks = (len - first) >> 4, len4 = len >> 1;
    const float4 *src[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        long f = f0 + 4 * j + r0;
        f = f < n_frames ? f : n_frames - 1;                        // rows past the end repeat the last frame (not stored)
        src[j] = reinterpret_cast<const float4 *>(frames) + f * len4 + (first >> 1) + col;
    }
    float4 q[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) q[j] = __ldg(src[j]);
    double pd = (double)acc0;
    for (int c = 0; c < n_chunks; ++c) {
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 8; ++j) tile[(4 * j + r0) * kPowPitch + col] = q[j];
        __syncwarp();
        if (c + 1 < n_chunks) {
#pragma unroll
            for (int j = 0; j < 8; ++j) q[j] = __ldg(src[j] + 8 * (c + 1));
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float4 v = tile[lane * kPowPitch + k];
            pd = power_step(pd, v.x, v.y, margin);
            pd = power_step(pd, v.z, v.w, margin);
        }
    }
    if (f0 + lane < n_frames) power[f0 + lane] = __fdiv_rn((float)pd, (float)len);
}
__global__ void __launch_bounds__(kThreads) k_frame_power_fast(const float2 *__restrict__ frames, float *__restrict__ power,
                                                               long n_frames, int len)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (long f = (long)blockIdx.x * kWarpsPerBlock + warp; f < n_frames; f += (long)gridDim.x * kWarpsPerBlock) {
        const float2 *x = frames + f * len;
        float acc = 0.f;
        for (int i = lane; i < len; i += 32) { float2 s = x[i]; acc = fmaf(s.x, s.x, fmaf(s.y, s.y, acc)); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) power[f] = acc / (float)len;
    }
}

// ------------------------------------------------------------------ channel (stand-alone)
// Transmission_Over_Air OFDM.c:645-653 with per-frame power: y.re = x.re + (float)(sqrt((double)np)*g),
// y.im = x.im.  One warp per frame.
__device__ __forceinline__ void noise_slot(int n, int &blk, int &j)
{
    if (n < 32) { blk = n >> 2; j = n & 3; return; }
    int base, l;
    if (n < 160) { l = (n - 32) & 63; base = n < 96 ? 8 : 24; }
    else {
        int s = (n - 160) / 80; l = (n - 160) - 80 * s;
        if (l < 16) { blk = 40 + 20 * s + (l >> 2); j = l & 3; return; }
        l -= 16; base = 44 + 20 * s;
    }
    blk = base + (l & 7) + 8 * (l >> 5);
    j = (l >> 3) & 3;
}

template <bool EXACT>
__device__ __forceinline__ float add_noise(float xr, float g, double sigma_d, float sigma_f)
{
    if constexpr (EXACT) return __fadd_rn(xr, __double2float_rn(__dmul_rn(sigma_d, (double)g)));
    else return fmaf(sigma_f, g, xr);
}
// the same with sigma pre-scaled by 2^896 and the draw widened without the XU pipe (see f2d_scaled): identical bits
template <bool EXACT>
__device__ __forceinline__ float add_noise_s(float xr, float g, double sigma_scaled, float sigma_f)
{
    if constexpr (EXACT) return __fadd_rn(xr, __double2float_rn(__dmul_rn(sigma_scaled, f2d_scaled(g))));
    else return fmaf(sigma_f, g, xr);
}

// Philox noise for buffers that are not LTS||data frames (e.g. the oversampled, repeated waveform): consecutive
// quadruples of samples share a block, domain 3.  One thread per block of four samples.
template <bool EXACT>
__global__ void __launch_bounds__(kThreads) k_awgn_philox_flat(const float2 *__restrict__ tx, const float *__restrict__ power, float snr_lin,
                                                               uint32_t seed, uint32_t stream, uint64_t frame0, float2 *__restrict__ ota,
                                                               long n_frames, int len)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (long f = (long)blockIdx.x * kWarpsPerBlock + warp; f < n_frames; f += (long)gridDim.x * kWarpsPerBlock) {
        const float np = __fdiv_rn(power[f], snr_lin);
        const double sigma_d = __dsqrt_rn((double)np);
        const float sigma_f = (float)sigma_d;
        const float2 *x = tx + f * len;
        float2 *y = ota + f * len;
        const bool vec = ((len & 1) == 0) && ((reinterpret_cast<uintptr_t>(tx) | reinterpret_cast<uintptr_t>(ota)) % 16 == 0);
        for (int b = lane; 4 * b < len; b += 32) {                 // one Philox block = four consecutive samples
            float z[4];
            philox_normals4(seed, stream, frame0 + (uint64_t)f, (uint32_t)b, 3u, z);
            const int n = 4 * b;
            if (vec && n + 3 < len) {                              // two 16-byte accesses instead of four 8-byte ones
                float4 a = *reinterpret_cast<const float4 *>(x + n), c = *reinterpret_cast<const float4 *>(x + n + 2);
                a.x = add_noise<EXACT>(a.x, z[0], sigma_d, sigma_f); a.z = add_noise<EXACT>(a.z, z[1], sigma_d, sigma_f);
                c.x = add_noise<EXACT>(c.x, z[2], sigma_d, sigma_f); c.z = add_noise<EXACT>(c.z, z[3], sigma_d, sigma_f);
                *reinterpret_cast<float4 *>(y + n) = a; *reinterpret_cast<float4 *>(y + n + 2) = c;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (n + j < len) {
                        float2 s = x[n + j];
                        s.x = add_noise<EXACT>(s.x, z[j], sigma_d, sigma_f);
                        y[n + j] = s;
                    }
                }
            }
        }
    }
}

template <bool EXACT, int NOISE>
__global__ void __launch_bounds__(kThreads) k_awgn(const float2 *__restrict__ tx, const float *__restrict__ g,
                                                   const float *__restrict__ power, float snr_lin, uint32_t seed,
                                                   uint32_t stream, uint64_t frame0, float2 *__restrict__ ota,
                                                   long n_frames, int len)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (long f = (long)blockIdx.x * kWarpsPerBlock + warp; f < n_frames; f += (long)gridDim.x * kWarpsPerBlock) {
        float np = __fdiv_rn(power[f], snr_lin);                // :647
        double sigma_d = __dsqrt_rn((double)np);                // sqrt(noise_power) in double, :651
        float sigma_f = (float)sigma_d;
        const float2 *x = tx + f * len;
        float2 *y = ota + f * len;
        for (int n = lane; n < len; n += 32) {
            float2 s = x[n];
            float gn;
            if (NOISE == kNoiseInject) gn = g[f * len + n];
            else {
                int blk, j; noise_slot(n, blk, j);
                float z[4];
                philox_normals4(seed, stream, frame0 + (uint64_t)f, (uint32_t)blk, kDomainNoise, z);
                gn = j == 0 ? z[0] : (j == 1 ? z[1] : (j == 2 ? z[2] : z[3]));
            }
            s.x = add_noise<EXACT>(s.x, gn, sigma_d, sigma_f);
            y[n] = s;
        }
    }
}

// z[j] without indexing a local array (selects stay in registers)
__device__ __forceinline__ float pick4(const float (&z)[4], int j) { return j == 0 ? z[0] : (j == 1 ? z[1] : (j == 2 ? z[2] : z[3])); }

// The channel of ofdm_awgn_philox_ex on LTS||data frames (include/ofdm_b200.h, DESIGN.md "Channels").  Noise power per frame:
// power[f] / snr_lin (the reference's definition), or np_fixed for every frame when power is NULL (Es/N0, Eb/N0).  Real rail:
// all of it on I, sigma = sqrt(np); COMPLEX: half per rail, sigma = sqrt(np / 2), the Q-rail draw is the normal in the same
// slot of domain 4.  EXACT: x + (float)(sigma_d * (double)g) per rail; fast: fmaf with sigma in fp32.  One warp per frame.
template <bool EXACT, bool COMPLEX>
__global__ void __launch_bounds__(kThreads) k_awgn_channel(const float2 *__restrict__ tx, const float *__restrict__ power,
                                                           float snr_lin, float np_fixed, uint32_t seed, uint32_t stream,
                                                           uint64_t frame0, float2 *__restrict__ ota, long n_frames, int len)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (long f = (long)blockIdx.x * kWarpsPerBlock + warp; f < n_frames; f += (long)gridDim.x * kWarpsPerBlock) {
        const float np = power ? __fdiv_rn(power[f], snr_lin) : np_fixed;
        const double sigma_d = __dsqrt_rn(COMPLEX ? __dmul_rn(0.5, (double)np) : (double)np);
        const float sigma_f = (float)sigma_d;
        const uint64_t fr = frame0 + (uint64_t)f;
        const float2 *x = tx + f * len;
        float2 *y = ota + f * len;
        for (int n = lane; n < len; n += 32) {
            float2 s = x[n];
            int blk, j; noise_slot(n, blk, j);
            float z[4];
            philox_normals4(seed, stream, fr, (uint32_t)blk, kDomainNoise, z);
            s.x = add_noise<EXACT>(s.x, pick4(z, j), sigma_d, sigma_f);
            if (COMPLEX) {
                philox_normals4(seed, stream, fr, (uint32_t)blk, kDomainNoiseQ, z);
                s.y = add_noise<EXACT>(s.y, pick4(z, j), sigma_d, sigma_f);
            }
            y[n] = s;
        }
    }
}

// ------------------------------------------------------------------ receiver (optionally fused with the channel)
struct RxParams {
    const float2 *in;           // OTA frames (NOISE == none) or TX frames (noise added in registers)
    const float *g;             // injected normals
    const float *power;         // per-frame mean power
    const uint32_t *tx_bits;
    long n_frames;
    int n_sym;
    float snr_lin;
    float radius_scale;         // kArithChecked: error-radius factor (kRadius; infinity forces every frame to be replayed)
    float radius_chan;          // kArithChecked: kChanRadius * sqrt(frame_len * snr_lin): times sigma = the speculated channel's share
    float evm_guard;            // EVM guard in radii (kEvmGuard; option "evm_guard")
    uint32_t seed, stream;
    uint64_t frame0;
    ofdm_counters *counters;
    unsigned long long *replayed;   // the context's count of exactly replayed frames (speculating kernels)
    ofdm_rx_dump dump;
};

// libgcc __divsc3 as gcc 13 builds it: quotient formula in double, one rounding to float, plus its
// zero-denominator recovery.  OFDM.c:1050
//
// sc is the 0.5*L factor the estimate was scaled with.  The kernels form H as (A+B)*sc, which equals the
// reference's 0.5*(A+B)*conj(L) (:848) in value but not in the sign of a zero; the recovery branch looks at
// the sign of a zero real part, so it is rebuilt there: with hr = 0.5*(A.x+B.x), hi = 0.5*(A.y+B.y), L = (lr, -0)
// the reference computes hr*lr - hi*(-0) = (hr*lr) + (hi*0), which is -0 only when both terms are -0.
__device__ __forceinline__ float2 div_exact(float2 n, float2 h, float sc)
{
    double a = n.x, b = n.y, c = h.x, d = h.y;
    double den = __dadd_rn(__dmul_rn(c, c), __dmul_rn(d, d));
    double x = __ddiv_rn(__dadd_rn(__dmul_rn(a, c), __dmul_rn(b, d)), den);
    double y = __ddiv_rn(__dsub_rn(__dmul_rn(b, c), __dmul_rn(a, d)), den);
    if (isnan(x) && isnan(y) && den == 0.0 && (!isnan(a) || !isnan(b))) {
        const bool lneg = sc < 0.f;
        const bool c_neg = signbit(h.x) && (signbit(h.y) != lneg);
        double inf = c_neg ? -(double)INFINITY : (double)INFINITY;
        x = __dmul_rn(inf, a); y = __dmul_rn(inf, b);
    }
    return make_float2(__double2float_rn(x), __double2float_rn(y));
}
__device__ __forceinline__ float2 div_fast(float2 n, float2 h)
{
    float inv = 1.0f / fmaf(h.x, h.x, h.y * h.y);
    return make_float2(fmaf(n.x, h.x, n.y * h.y) * inv, fmaf(n.y, h.x, -n.x * h.y) * inv);
}

// One data bin through equalise :1050, slicer :860-868, demod :883-902, BER :1158 and the EVM terms :1114
// for the dump path (every value materialised, exact division in EXACT mode).
// Returns the rail-error flags (bit0 = I rail, bit1 = Q rail).
template <bool EXACT>
__device__ __forceinline__ uint32_t process_bin_full(float2 F, float2 Hh, float sc, uint32_t txp, float &e2, float2 &E, bool &re_pos, bool &im_pos)
{
    E = EXACT ? div_exact(F, Hh, sc) : div_fast(F, Hh);
    re_pos = E.x > 0.f; im_pos = E.y > 0.f;
    const uint32_t A = txp & 1u, B = txp >> 1;
    const bool i_pos = (A ^ B) == 0u, q_pos = A == 0u;           // tx rails, QPSK_Modulator :423-430
    const float er = E.x - (i_pos ? kQpsk : -kQpsk), ei = E.y - (q_pos ? kQpsk : -kQpsk);
    e2 = fmaf(er, er, fmaf(ei, ei, e2));
    return (uint32_t)(re_pos != i_pos) | ((uint32_t)(im_pos != q_pos) << 1);
}

// The sweep path's version of the same bin.  Returns the rail errors packed for cheap accumulation:
// bits 0..7 += I-rail error, 8..15 += Q-rail error, 16..23 += both.  (Bit errors follow from the
// non-Gray map, SURVEY Q5: a Q error flips bit a, bit b flips when exactly one rail is wrong.)
//
// EXACT: the decision the reference takes is the sign of float(num/den) (:1050, :860).  For normal
// magnitudes that is the sign of the exact numerator a*c+b*d (resp. b*c-a*d).  Its fp32 evaluation
// errs by < 2^-23 m, m = (|a|+|b|)(|c|+|d|), and is trusted only above max(1e-6 m, 1e-30) (which also keeps m >= 1e-30,
// so denormal products cannot matter) with den < 1e14 (the float quotient then stays above the denormal range);
// every other case (about 1e-6 of the bins, plus degenerate frames) takes the exact double-widened
// division.  The EVM term uses the fp32 quotient (1e-5 contract).
template <bool EXACT>
__device__ __forceinline__ uint32_t process_bin_hot(float2 F, float2 Hh, float sc, uint32_t txp, bool valid, float &e2)
{
    const float a = F.x, b = F.y, c = Hh.x, d = Hh.y;
    // numerator F * conj(H) = (fma(a, c, b*d), fma(b, c, -(a*d))): FMUL2 with a broadcast + FFMA2 with a mixed-sign addend
    const float2 pt = __fmul2_rn(make_float2(d, d), make_float2(b, a));
    const float2 S = __ffma2_rn(make_float2(c, c), F, make_float2(pt.x, -pt.y));
    const float sr = S.x, si = S.y;
    const float den = fmaf(c, c, d * d);
    float inv;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(den));
    float2 E = __fmul2_rn(S, make_float2(inv, inv));
    const uint32_t sq = txp << 31, sx = (txp ^ (txp >> 1)) << 31;          // IEEE sign bits of the tx Q / I rails
    uint32_t ei_ = (__float_as_uint(sr) ^ sx) >> 31, eq_ = (__float_as_uint(si) ^ sq) >> 31;
    if (EXACT) {
        // |num| > max(1e-6 m, 1e-30) also bounds m from below (|num| <= m), den < 1e14 keeps the float quotient above the
        // denormal range; non-finite m or den fail the comparisons.
        const float m = (fabsf(a) + fabsf(b)) * (fabsf(c) + fabsf(d));
        const bool safe = fminf(fabsf(sr), fabsf(si)) > fmaxf(1e-6f * m, 1e-30f) && den < 1e14f;
        if (!safe && valid) {
            E = div_exact(F, Hh, sc);
            ei_ = (uint32_t)((E.x > 0.f) != (sx == 0u));
            eq_ = (uint32_t)((E.y > 0.f) != (sq == 0u));
        }
    }
    // E - tx point: the tx rails are +-1/sqrt(2) = 0x3F3504F3 with the sign bits above
    const float2 D = __fadd2_rn(E, make_float2(__uint_as_float(0xBF3504F3u ^ sx), __uint_as_float(0xBF3504F3u ^ sq)));
    const float t = fmaf(D.x, D.x, D.y * D.y);
    e2 += valid ? t : 0.f;
    const uint32_t pk = ei_ | (eq_ << 8) | ((ei_ & eq_) << 16);
    return valid ? pk : 0u;
}

// Fused receiver.  DUMP = false is the sweep path: totals only; the bins of the two first data
// symbols are shared with the (otherwise idle) LTS lane groups so all 32 lanes work through the
// decision stage.  DUMP = true writes any of the per-bin / per-frame outputs, always dividing exactly.
template <bool EXACT, int NOISE, bool DUMP>
__global__ void __launch_bounds__(kThreads, DUMP ? 1 : 2) k_rx_frames(RxParams p)
{
    __shared__ float2 s_tile[kWarpsPerBlock][kWarpTile];
    __shared__ float2 s_lts[kWarpsPerBlock][2][72];
    __shared__ unsigned long long s_cnt[kWarpsPerBlock][4];
    __shared__ double s_sum[kWarpsPerBlock][2];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, u = lane & 7;
    const uint32_t grp_mask = 0xFFu << (grp * 8);
    float2 *tile = s_tile[warp] + grp * kGroupPitch;
    const float2 *ltsA = s_lts[warp][0], *ltsB = s_lts[warp][1];
    Tw<EXACT> tw; tw.load(u);
    // per-lane bin info for natural bins u + 8j: data index byte (>= 0x80: null / pilot) and the L sign
    uint32_t dlo = 0, dhi = 0, lneg = 0, lnul = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const uint32_t d = (uint32_t)(uint8_t)c_tab.bin_data[u + 8 * j];
        if (j < 4) dlo |= d << (8 * j); else dhi |= d << (8 * (j - 4));
        const int l = c_tab.bin_lts[u + 8 * j];
        lneg |= (uint32_t)(l < 0) << j; lnul |= (uint32_t)(l == 0) << j;
    }
    // H = 0.5*(A+B)*conj(L), :848; L is real so the scaling is exact in float
    auto h_of = [&](int j) {
        const float2 A = ltsA[u + 8 * j], B = ltsB[u + 8 * j];
        const float sc = ((lnul >> j) & 1u) ? 0.f : (((lneg >> j) & 1u) ? -0.5f : 0.5f);
        return make_float2(__fmul_rn(__fadd_rn(A.x, B.x), sc), __fmul_rn(__fadd_rn(A.y, B.y), sc));
    };
    auto sc_of = [&](int j) { return ((lnul >> j) & 1u) ? 0.f : (((lneg >> j) & 1u) ? -0.5f : 0.5f); };
    const int n_sym = p.n_sym, len = 160 + 80 * n_sym;
    const int n_pass = 1 + (n_sym > 2 ? (n_sym - 2 + 3) / 4 : 0);
    const double q = (double)kQpsk;
    const double ref2_frame = 48.0 * n_sym * (2.0 * q * q);     // sum |tx|^2 over the frame's data bins
    const float inv_ref2 = (float)(1.0 / ref2_frame);
    const long stride = (long)gridDim.x * kWarpsPerBlock;
    const long f_first = (long)blockIdx.x * kWarpsPerBlock + warp;

    uint32_t a_i = 0, a_q = 0, a_both = 0, a_ferr = 0, a_frames = 0;   // per lane
    double a_e2 = 0.0, a_evm = 0.0;                                     // warp-uniform

    for (long f_chunk = f_first; f_chunk < p.n_frames; f_chunk += 32 * stride) {
        // lane l prepares sigma = sqrt((double)(P / snr_lin)) (:647, :651) of the chunk's l-th frame
        double sig_mine = 0.0;
        if (NOISE != kNoiseNone) {
            const long fl = f_chunk + lane * stride;
            if (fl < p.n_frames) sig_mine = __dsqrt_rn((double)__fdiv_rn(p.power[fl], p.snr_lin));
        }
        float c_e2 = 0.f, c_evm = 0.f;
        for (int k = 0; k < 32; ++k) {
            const long f = f_chunk + k * stride;
            if (f >= p.n_frames) break;
            const float2 *x = p.in + f * len;
            const double sigma_d = NOISE != kNoiseNone ? __shfl_sync(0xffffffffu, sig_mine, k) : 0.0;
            const float sigma_f = (float)sigma_d;
            uint32_t f_i = 0, f_q = 0, f_both = 0;
            float f_e2 = 0.f;
            for (int pass = 0; pass < n_pass; ++pass) {
                const int sym = pass == 0 ? grp - 2 : 2 + (pass - 1) * 4 + grp;     // < 0: LTS half
                const bool active = sym < n_sym;
                const int n0 = sym < 0 ? 32 + 64 * grp : 176 + 80 * sym;           // Channel_Estimation :837-838, CP strip :1028
                float2 v[8];
                float z[8];
                if (NOISE == kNoisePhilox && active) {
                    const int base = window_block_base(n0) + u;
                    float za[4], zb[4];
                    philox_normals4(p.seed, p.stream, p.frame0 + (uint64_t)f, (uint32_t)base, kDomainNoise, za);
                    philox_normals4(p.seed, p.stream, p.frame0 + (uint64_t)f, (uint32_t)(base + 8), kDomainNoise, zb);
#pragma unroll
                    for (int m = 0; m < 4; ++m) { z[m] = za[m]; z[4 + m] = zb[m]; }
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int m = slot_m<EXACT>(i);
                    float2 s = make_float2(0.f, 0.f);
                    if (active) {
                        s = x[n0 + u + 8 * m];
                        if (NOISE == kNoiseInject) s.x = add_noise<EXACT>(s.x, p.g[f * len + n0 + u + 8 * m], sigma_d, sigma_f);
                        if (NOISE == kNoisePhilox) s.x = add_noise<EXACT>(s.x, z[m], sigma_d, sigma_f);
                    }
                    v[i] = s;
                }
                fft64<EXACT>(v, tw, tile, u);                                       // natural bins u + 8j
                if (pass == 0) {
                    if (grp < 2) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) s_lts[warp][grp][u + 8 * j] = v[j];
                    }
                    __syncwarp();
                    if (DUMP && p.dump.H != nullptr && grp == 0) {
                        float2 *Hout = reinterpret_cast<float2 *>(p.dump.H) + f * 64;
#pragma unroll
                        for (int j = 0; j < 8; ++j) Hout[(u + 8 * j + 32) & 63] = h_of(j);
                    }
                }
                if (!DUMP && pass == 0) {
                    // lanes of LTS group g take over slots 4..7 of data group g+2 (the same symbol g)
                    const int dsym = grp & 1, off = grp < 2 ? 4 : 0;
                    const uint32_t dsel = grp < 2 ? dhi : dlo;
                    const uint32_t *w = p.tx_bits + (f * n_sym + dsym) * 3;
                    uint32_t w0 = 0, w1 = 0, w2 = 0;
                    if (dsym < n_sym) { w0 = w[0]; w1 = w[1]; w2 = w[2]; }
                    uint32_t pk = 0;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const float wx = __shfl_down_sync(0xffffffffu, v[4 + kk].x, 16), wy = __shfl_down_sync(0xffffffffu, v[4 + kk].y, 16);
                        const float2 X = grp < 2 ? make_float2(wx, wy) : v[kk];
                        const uint32_t d = (dsel >> (8 * kk)) & 0xFFu;
                        pk += process_bin_hot<EXACT>(X, h_of(off + kk), sc_of(off + kk), bit_pair(w0, w1, w2, (int)d), d < 0x80u && dsym < n_sym, f_e2);
                    }
                    f_i += pk & 0xFFu; f_q += (pk >> 8) & 0xFFu; f_both += pk >> 16;
                } else if (!DUMP) {
                    const int ssym = active ? sym : 0;
                    const uint32_t *w = p.tx_bits + (f * n_sym + ssym) * 3;
                    const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
                    uint32_t pk = 0;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const uint32_t d = ((j < 4 ? dlo : dhi) >> (8 * (j & 3))) & 0xFFu;
                        pk += process_bin_hot<EXACT>(v[j], h_of(j), sc_of(j), bit_pair(w0, w1, w2, (int)d), d < 0x80u && active, f_e2);
                    }
                    f_i += pk & 0xFFu; f_q += (pk >> 8) & 0xFFu; f_both += pk >> 16;
                } else if (active && sym >= 0) {
                    const uint32_t *w = p.tx_bits + (f * n_sym + sym) * 3;
                    const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
                    uint32_t o0 = 0, o1 = 0, o2 = 0;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const uint32_t d = ((j < 4 ? dlo : dhi) >> (8 * (j & 3))) & 0xFFu;
                        if (d >= 0x80u) continue;                                   // demap :1063-1068 keeps the 48 data bins
                        float2 E; bool rp, ip;
                        const uint32_t e = process_bin_full<EXACT>(v[j], h_of(j), sc_of(j), bit_pair(w0, w1, w2, (int)d), f_e2, E, rp, ip);
                        f_i += e & 1u; f_q += e >> 1; f_both += (e == 3u);
                        if (p.dump.eq != nullptr) reinterpret_cast<float2 *>(p.dump.eq)[(f * n_sym + sym) * 48 + d] = E;
                        if (p.dump.sliced != nullptr)
                            reinterpret_cast<float2 *>(p.dump.sliced)[(f * n_sym + sym) * 48 + d] =
                                make_float2(rp ? kQpsk : -kQpsk, ip ? kQpsk : -kQpsk);
                        const uint32_t sh = demod_pair(rp, ip) << (2 * (d & 15u));
                        if (d < 16u) o0 |= sh; else if (d < 32u) o1 |= sh; else o2 |= sh;
                    }
                    if (p.dump.bits != nullptr) {
#pragma unroll
                        for (int o = 1; o < 8; o <<= 1) {
                            o0 |= __shfl_xor_sync(grp_mask, o0, o);
                            o1 |= __shfl_xor_sync(grp_mask, o1, o);
                            o2 |= __shfl_xor_sync(grp_mask, o2, o);
                        }
                        if (u == 0) { uint32_t *ob = p.dump.bits + (f * n_sym + sym) * 3; ob[0] = o0; ob[1] = o1; ob[2] = o2; }
                    }
                }
                __syncwarp();
            }
            // bit errors of a bin = q_err + (i_err xor q_err) = i + 2q - 2*both   (BER :1158 under the map of :423-430)
            const uint32_t f_bit_lane = f_i + 2u * f_q - 2u * f_both;
            const bool any_err = __any_sync(0xffffffffu, f_bit_lane != 0u);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) f_e2 += __shfl_xor_sync(0xffffffffu, f_e2, o);
            const float evm = sqrtf(f_e2 * inv_ref2);                               // :1124
            if (DUMP) {
                const uint32_t f_bit = warp_sum(f_bit_lane);
                if (lane == 0) {
                    if (p.dump.frame_bit_errors != nullptr) p.dump.frame_bit_errors[f] = (int32_t)f_bit;
                    if (p.dump.frame_evm_lin != nullptr) p.dump.frame_evm_lin[f] = evm;
                }
            }
            a_i += f_i; a_q += f_q; a_both += f_both;
            a_ferr += any_err; a_frames += 1;
            c_e2 += f_e2; c_evm += evm;
        }
        a_e2 += (double)c_e2; a_evm += (double)c_evm;
    }
    if (p.counters == nullptr) return;
    const uint32_t t_i = warp_sum(a_i), t_q = warp_sum(a_q), t_both = warp_sum(a_both);
    if (lane == 0) {
        s_cnt[warp][0] = (unsigned long long)t_i + 2ull * t_q - 2ull * t_both;     // bit errors
        s_cnt[warp][1] = (unsigned long long)t_i + t_q;                             // rail errors
        s_cnt[warp][2] = a_ferr; s_cnt[warp][3] = a_frames;
        s_sum[warp][0] = a_e2; s_sum[warp][1] = a_evm;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long c[4] = {0, 0, 0, 0}; double s[2] = {0, 0};
        for (int w = 0; w < kWarpsPerBlock; ++w) {
            for (int k = 0; k < 4; ++k) c[k] += s_cnt[w][k];
            for (int k = 0; k < 2; ++k) s[k] += s_sum[w][k];
        }
        if (c[3] != 0) {
            ofdm_counters *o = p.counters;
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->bit_errors), c[0]);
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->rail_errors), c[1]);
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->frames_in_error), c[2]);
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->frames), c[3]);
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->bits), c[3] * 96ull * (unsigned long long)n_sym);
            atomicAdd(&o->sum_err2, s[0]);
            atomicAdd(&o->sum_ref2, (double)c[3] * ref2_frame);
            atomicAdd(&o->sum_evm_lin, s[1]);
        }
    }
}

// ------------------------------------------------------------------ stand-alone receiver stages
// The reference's receiver is a sequence of separate functions / inline blocks; the fused kernels above are what a
// sweep runs, these are their 1:1 batched counterparts (device buffers in, device buffers out) so that a caller can
// stop after any stage exactly as with the reference (SURVEY 8(b)).

// CP strip OFDM.c:1024-1031: frames [n][frame_len] -> symbol bodies [n][n_sym][64]; data_off = sample index of the
// first data symbol (160 for LTS || data frames, 320 with the STS slot in front as in the reference's own frame)
// (one warp per frame: 32 consecutive samples per access, no division per element)
__global__ void __launch_bounds__(kThreads) k_strip_cp(const float2 *__restrict__ frames, float2 *__restrict__ out, long n_frames, int n_sym, int frame_len, int data_off)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int per = n_sym * 64;
    for (long f = (long)blockIdx.x * kWarpsPerBlock + warp; f < n_frames; f += (long)gridDim.x * kWarpsPerBlock) {
        const float2 *x = frames + f * frame_len + data_off + 16;
        float2 *y = out + f * per;
        for (int idx = lane; idx < per; idx += 32) y[idx] = x[80 * (idx >> 6) + (idx & 63)];
    }
}

// Channel_Estimation OFDM.c:830-850: fft of the two LTS halves (samples lts_off + 32 .. + 95 and + 96 .. + 159 of each
// frame), H[c] = 0.5 * (A[c] + B[c]) * conj(L[c]) on the centred grid.  EXACT evaluates the product as gcc does for
// `double * float complex * float complex` -- (0.5 re, 0.5 im) then the full complex multiply by (L, -0) in double, one
// rounding to float -- so that even the signs of zeros (null bins, cancelling halves) are the reference's.
// A warp serves two frames: lane group 2k + h transforms half h of frame k.
template <bool EXACT>
__global__ void __launch_bounds__(kThreads) k_channel_estimate(const float2 *__restrict__ frames, float2 *__restrict__ H, long n_frames,
                                                               int frame_len, int lts_off)
{
    __shared__ float2 s_tile[kWarpsPerBlock][kWarpTile];
    __shared__ float2 s_b[kWarpsPerBlock][2][72];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, u = lane & 7;
    float2 *tile = s_tile[warp] + grp * kGroupPitch;
    Tw<EXACT> tw; tw.load(u);
    const long n_pairs = (n_frames + 1) / 2;
    for (long pr = (long)blockIdx.x * kWarpsPerBlock + warp; pr < n_pairs; pr += (long)gridDim.x * kWarpsPerBlock) {
        const long f = 2 * pr + (grp >> 1);
        const bool active = f < n_frames;
        const int n0 = lts_off + 32 + 64 * (grp & 1);
        float2 v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = active ? frames[f * frame_len + n0 + u + 8 * slot_m<EXACT>(i)] : make_float2(0.f, 0.f);
        fft64<EXACT>(v, tw, tile, u);
        if (grp & 1) {
#pragma unroll
            for (int j = 0; j < 8; ++j) s_b[warp][grp >> 1][u + 8 * j] = v[j];
        }
        __syncwarp();
        if (!(grp & 1) && active) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int p = u + 8 * j;
                const float2 B = s_b[warp][grp >> 1][p];
                const float l = (float)c_tab.bin_lts[p];
                float2 h;
                if (EXACT) {
                    const float sr = __fadd_rn(v[j].x, B.x), si = __fadd_rn(v[j].y, B.y);
                    const double hr = __dmul_rn(0.5, (double)sr), hi = __dmul_rn(0.5, (double)si), lr = (double)l, li = -0.0;
                    h.x = __double2float_rn(__dsub_rn(__dmul_rn(hr, lr), __dmul_rn(hi, li)));
                    h.y = __double2float_rn(__dadd_rn(__dmul_rn(hr, li), __dmul_rn(hi, lr)));
                } else {
                    h = make_float2((v[j].x + B.x) * (0.5f * l), (v[j].y + B.y) * (0.5f * l));
                }
                H[f * 64 + ((p + 32) & 63)] = h;
            }
        }
        __syncwarp();
    }
}

// libgcc __divsc3 (gcc 13: quotient formula in double, one rounding to float) with all three of its NaN recoveries
__device__ __forceinline__ float2 divsc3(float2 n, float2 h)
{
    double a = n.x, b = n.y, c = h.x, d = h.y;
    const double den = __dadd_rn(__dmul_rn(c, c), __dmul_rn(d, d));
    double x = __ddiv_rn(__dadd_rn(__dmul_rn(a, c), __dmul_rn(b, d)), den);
    double y = __ddiv_rn(__dsub_rn(__dmul_rn(b, c), __dmul_rn(a, d)), den);
    if (isnan(x) && isnan(y)) {
        const double inf = (double)INFINITY;
        if (c == 0.0 && d == 0.0 && (!isnan(a) || !isnan(b))) {
            x = __dmul_rn(copysign(inf, c), a); y = __dmul_rn(copysign(inf, c), b);
        } else if ((isinf(a) || isinf(b)) && isfinite(c) && isfinite(d)) {
            a = copysign(isinf(a) ? 1.0 : 0.0, a); b = copysign(isinf(b) ? 1.0 : 0.0, b);
            x = __dmul_rn(inf, __dadd_rn(__dmul_rn(a, c), __dmul_rn(b, d)));
            y = __dmul_rn(inf, __dsub_rn(__dmul_rn(b, c), __dmul_rn(a, d)));
        } else if ((isinf(c) || isinf(d)) && isfinite(a) && isfinite(b)) {
            c = copysign(isinf(c) ? 1.0 : 0.0, c); d = copysign(isinf(d) ? 1.0 : 0.0, d);
            x = __dmul_rn(0.0, __dadd_rn(__dmul_rn(a, c), __dmul_rn(b, d)));
            y = __dmul_rn(0.0, __dsub_rn(__dmul_rn(b, c), __dmul_rn(a, d)));
        }
    }
    return make_float2(__double2float_rn(x), __double2float_rn(y));
}

// one-tap equaliser OFDM.c:1044-1052: E[f][s][c] = F[f][s][c] / H[f][c] for all 64 centred bins (the 12 null bins
// come out as the inf / NaN the reference computes there and never reads -- SURVEY Q16)
// (one warp per frame: the estimate's two bins per lane are read once and serve all the frame's symbols)
template <bool EXACT>
__global__ void __launch_bounds__(kThreads) k_equalize(const float2 *__restrict__ F, const float2 *__restrict__ H, float2 *__restrict__ E, long n_frames, int n_sym)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (long f = (long)blockIdx.x * kWarpsPerBlock + warp; f < n_frames; f += (long)gridDim.x * kWarpsPerBlock) {
        const float2 h0 = H[f * 64 + lane], h1 = H[f * 64 + 32 + lane];
        const float2 *x = F + f * n_sym * 64;
        float2 *y = E + f * n_sym * 64;
        for (int s = 0; s < n_sym; ++s) {
            const float2 a = x[s * 64 + lane], b = x[s * 64 + 32 + lane];
            y[s * 64 + lane] = EXACT ? divsc3(a, h0) : div_fast(a, h0);
            y[s * 64 + 32 + lane] = EXACT ? divsc3(b, h1) : div_fast(b, h1);
        }
    }
}

// demap OFDM.c:1059-1069: the 48 data bins of each centred 64-grid, in order; column = data index d (block of 4 x 48 threads)
__global__ void __launch_bounds__(kRows4 * 48) k_demap(const float2 *__restrict__ grid, float2 *__restrict__ out, long n_sym_total)
{
    const int d = threadIdx.x % 48, r = threadIdx.x / 48;
    const int src = (c_tab.data_bin[d] + 32) & 63;
    for (long sym = (long)blockIdx.x * kRows4 + r; sym < n_sym_total; sym += (long)gridDim.x * kRows4)
        out[sym * 48 + d] = grid[sym * 64 + src];
}

// AGC_Receiver OFDM.c:852-871: the hard-decision slicer -- each rail to +1/sqrt(2) if > 0 else -1/sqrt(2) (0 and NaN go negative)
__global__ void k_agc_slicer(const float2 *__restrict__ in, float2 *__restrict__ out, long n_points)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_points) return;
    const float2 z = in[i];
    out[i] = make_float2(z.x > 0.f ? kQpsk : -kQpsk, z.y > 0.f ? kQpsk : -kQpsk);
}
// the same on 16-byte aligned buffers: two points per access, grid-stride
__global__ void __launch_bounds__(kThreads) k_agc_slicer2(const float4 *__restrict__ in, float4 *__restrict__ out, long n_pairs)
{
    for (long i = (long)blockIdx.x * kThreads + threadIdx.x; i < n_pairs; i += (long)gridDim.x * kThreads) {
        const float4 z = in[i];
        out[i] = make_float4(z.x > 0.f ? kQpsk : -kQpsk, z.y > 0.f ? kQpsk : -kQpsk, z.z > 0.f ? kQpsk : -kQpsk, z.w > 0.f ? kQpsk : -kQpsk);
    }
}

// QPSK_Demodulator OFDM.c:873-908 with the reference's own comparisons: (+,+) -> 00, (-,+) -> 01, (-,-) -> 10, anything else
// (a zero or NaN rail included) -> 11; bit 2j = c, bit 2j+1 = d.  One thread per packed word (16 points).
__device__ __forceinline__ uint32_t demod_point(float a, float b)
{
    uint32_t c, d;
    if (a > 0.f && b > 0.f) { c = 0; d = 0; }
    else if (a < 0.f && b > 0.f) { c = 0; d = 1; }
    else if (a < 0.f && b < 0.f) { c = 1; d = 0; }
    else { c = 1; d = 1; }
    return c | (d << 1);
}
// 16-byte aligned input: a warp turns 512 points (4 KB, coalesced 16-byte loads) into 32 words.  Load k of a lane holds points
// 64 k + 2 lane and + 1, i.e. bits 4 (lane & 7) .. + 3 of word 4 k + (lane >> 3); the eight lanes of a group OR their nibbles.
__global__ void __launch_bounds__(kThreads) k_qpsk_demod_warp(const float4 *__restrict__ in, uint32_t *__restrict__ bits, long n_words)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long n_chunks = (n_words + 31) / 32;
    for (long ch = (long)blockIdx.x * kWarpsPerBlock + warp; ch < n_chunks; ch += (long)gridDim.x * kWarpsPerBlock) {
        const float4 *src = in + ch * 256 + lane;                    // 256 float4 = 512 points per chunk
        uint32_t mine = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const long w = ch * 32 + 4 * k + (lane >> 3);
            uint32_t v = 0;
            if (w < n_words) {
                const float4 z = src[32 * k];
                v = (demod_point(z.x, z.y) | (demod_point(z.z, z.w) << 2)) << (4 * (lane & 7));
            }
            v |= __shfl_xor_sync(0xffffffffu, v, 1);
            v |= __shfl_xor_sync(0xffffffffu, v, 2);
            v |= __shfl_xor_sync(0xffffffffu, v, 4);
            // word 4 k + g is complete in the lanes of group g: lane 4 k + g keeps it, so that lane L ends up with word L of the chunk
            const uint32_t got = __shfl_sync(0xffffffffu, v, 8 * (lane & 3));
            if ((lane >> 2) == k) mine = got;
        }
        const long w = ch * 32 + lane;
        if (w < n_words) bits[w] = mine;
    }
}
__global__ void k_qpsk_demod(const float2 *__restrict__ in, uint32_t *__restrict__ bits, long n_words)
{
    const long w = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_words) return;
    const float2 *z = in + w * 16;
    uint32_t v = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const float a = z[j].x, b = z[j].y;
        uint32_t c, d;
        if (a > 0.f && b > 0.f) { c = 0; d = 0; }
        else if (a < 0.f && b > 0.f) { c = 0; d = 1; }
        else if (a < 0.f && b < 0.f) { c = 1; d = 0; }
        else { c = 1; d = 1; }
        v |= (c | (d << 1)) << (2 * j);
    }
    bits[w] = v;
}

}  // namespace ofdm
