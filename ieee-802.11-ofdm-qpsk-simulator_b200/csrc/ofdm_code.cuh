// ofdm_code.cuh -- the 802.11a convolutional code on the coded link (DESIGN.md section 6.2): k_conv_encode (encoder, tail,
// puncturing, interleaver and Gray precoding in one pass) and k_viterbi (64-state maximum-likelihood decoder over the whole
// tail-terminated frame, fed by the receiver's H and eq dumps).
#pragma once
#include "ofdm_kernels.cuh"

namespace ofdm {

constexpr int kCodeR12 = 1, kCodeR34 = 2;
constexpr int kDecisionSoft = 0, kDecisionHard = 1;
constexpr uint32_t kG0 = 0133, kG1 = 0171;        // generators, octal: window bit 6 = newest input bit, bit 0 = the oldest
constexpr int kVitWarps = 8;                      // k_viterbi: warps per block, one frame per warp
constexpr int kVitSmemMax = 96 * 1024;            // survivors of a block up to this size live in shared memory, beyond in HBM

__host__ __device__ constexpr int code_dbps(int rate) { return rate == kCodeR12 ? 48 : 72; }   // data bits per OFDM symbol
// 802.11a interleaver for N_CBPS = 96, N_BPSC = 2: coded bit k of a symbol -> position i (i >> 1 = data point, i & 1 = Q rail)
__host__ __device__ constexpr int ilv_pos(int k) { return 6 * (k & 15) + (k >> 4); }

__device__ __forceinline__ uint32_t parity(uint32_t v) { return __popc(v) & 1u; }

// One thread per (frame, OFDM symbol): the symbol's N_DBPS input bits, preceded by the 6 bits before them (the encoder state),
// are fed through the K = 7 shift register; bits at or beyond K_info = n_sym N_DBPS - 6 are the zero tail.  The 96 coded
// bits (A before B; rate 3/4 sends A0 B0 A1 B2 of every 3 input bits) go through the interleaver, and each data point's pair
// (c0 on I, c1 on Q) becomes payload bits (2d, 2d+1) = (!c1, c0 ^ c1), which the transmitter's map sends as
// I = (2 c0 - 1)/sqrt(2), Q = (2 c1 - 1)/sqrt(2).  Consecutive threads write consecutive 12-byte triples.
template <int RATE>
__global__ void __launch_bounds__(256) k_conv_encode(const uint32_t *__restrict__ info, uint32_t *__restrict__ payload, long n_frames, int n_sym)
{
    constexpr int N = code_dbps(RATE);
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_frames * n_sym) return;
    const long f = t / n_sym;
    const int s = (int)(t - f * n_sym);
    const int k_info = n_sym * N - 6;
    const uint32_t *in = info + f * n_sym * 3;
    long word_idx = -1;
    uint32_t word = 0, win = 0;
    uint32_t cb[3] = {0u, 0u, 0u};
#pragma unroll
    for (int j = -6; j < N; ++j) {
        const int b = s * N + j;                                // flat bit index within the frame
        uint32_t x = 0u;
        if (b >= 0 && b < k_info) {
            if ((b >> 5) != word_idx) { word_idx = b >> 5; word = in[word_idx]; }
            x = (word >> (b & 31)) & 1u;
        }
        win = (win >> 1) | (x << 6);
        if (j < 0) continue;
        const uint32_t a = parity(win & kG0), bb = parity(win & kG1);
        if (RATE == kCodeR12) {
            cb[(2 * j) >> 5] |= a << ((2 * j) & 31);
            cb[(2 * j + 1) >> 5] |= bb << ((2 * j + 1) & 31);
        } else {
            const int g = j / 3, r = j % 3, k = 4 * g;
            if (r == 0) { cb[k >> 5] |= a << (k & 31); cb[(k + 1) >> 5] |= bb << ((k + 1) & 31); }
            else if (r == 1) cb[(k + 2) >> 5] |= a << ((k + 2) & 31);
            else cb[(k + 3) >> 5] |= bb << ((k + 3) & 31);
        }
    }
    uint32_t r[3] = {0u, 0u, 0u};
#pragma unroll
    for (int k = 0; k < 96; ++k) {
        const int i = ilv_pos(k);
        r[i >> 5] |= ((cb[k >> 5] >> (k & 31)) & 1u) << (i & 31);
    }
    uint32_t *out = payload + t * 3;
#pragma unroll
    for (int w = 0; w < 3; ++w) {
        const uint32_t e = r[w] & 0x55555555u, o = (r[w] >> 1) & 0x55555555u;          // c0 (I rail), c1 (Q rail) per point
        out[w] = (~o & 0x55555555u) | ((e ^ o) << 1);
    }
}

struct VitParams {
    const float2 *H;          // [frames][64] centred channel estimate
    const float2 *eq;         // [frames][n_sym * 48] equalised data points
    const uint32_t *info;     // [frames][n_sym * 3] information words (nullable)
    uint32_t *decoded;        // [frames][n_sym * 3] (nullable)
    uint2 *surv_global;       // survivors in HBM: [grid warps][n_sym * N_DBPS] (null: in shared memory)
    ofdm_counters *counters;  // nullable
    long n_frames;
    int n_sym;
};

inline size_t vit_surv_bytes(int rate, int n_sym) { return (size_t)n_sym * code_dbps(rate) * sizeof(uint2); }

// decoder input of one rail of a data point: soft L = w eq_rail with w = |H|^2 (the CSI-weighted zero-forcing value), hard
// L = +-1 by the slicer's rule (0 and NaN negative); a non-finite L is an erasure
template <int DECISION>
__device__ __forceinline__ float vit_input(float w, float e)
{
    if (DECISION == kDecisionHard) return e > 0.f ? 1.f : -1.f;
    const float l = __fmul_rn(w, e);
    return fabsf(l) < INFINITY ? l : 0.f;          // NaN and +-inf: erasure
}

// One frame per warp, lane j owning states j and j + 32.  A trellis step is the butterfly {2j, 2j+1} -> {j, j+32}: the old
// metrics come through four shuffles, both candidates of a new state are compared (the higher index wins only if strictly
// larger), the 64 decision bits are two ballots, and every new metric has the new metric of state 0 subtracted.  Per symbol the
// warp first turns eq and H into the 96 interleaved decoder inputs and the N_DBPS depunctured (A, B) pairs in shared memory.
// The survivors (8 bytes a step) are buffered one per lane and stored 32 steps at a time, to shared memory or to HBM; the
// traceback runs on the whole warp from state 0, 32 steps per coalesced load, one decoded word per 32 steps.
template <int RATE, int DECISION>
__global__ void __launch_bounds__(kVitWarps * 32, 1) k_viterbi(const VitParams p)
{
    constexpr int N = code_dbps(RATE);
    extern __shared__ uint2 s_surv[];
    __shared__ float s_li[kVitWarps][96];
    __shared__ float2 s_pair[kVitWarps][N];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_sym = p.n_sym, T = n_sym * N, k_info = T - 6, n_words = n_sym * 3;
    const long gwarp = (long)blockIdx.x * kVitWarps + warp;
    uint2 *surv = p.surv_global ? p.surv_global + gwarp * T : s_surv + (long)warp * T;
    // branch signs of the transition (state 2 lane, input 0); the three other transitions of the butterfly are their negation
    // or themselves (both generators tap the newest and the oldest bit)
    const float sa = parity((2u * lane) & kG0) ? 1.f : -1.f, sb = parity((2u * lane) & kG1) ? 1.f : -1.f;
    const int src = (2 * lane) & 31;
    const int d_hi = lane + 32;                                  // second data point of the lane (< 48 on lanes 0..15)
    const int c_lo = (c_tab.data_bin[lane] + 32) & 63, c_hi = lane < 16 ? (c_tab.data_bin[d_hi] + 32) & 63 : 0;
    uint32_t a_err = 0, a_ferr = 0, a_frames = 0;

    for (long f = gwarp; f < p.n_frames; f += (long)gridDim.x * kVitWarps) {
        float w_lo = 0.f, w_hi = 0.f;
        if (DECISION == kDecisionSoft) {
            const float2 h0 = p.H[f * 64 + c_lo];
            w_lo = __fadd_rn(__fmul_rn(h0.x, h0.x), __fmul_rn(h0.y, h0.y));
            if (lane < 16) {
                const float2 h1 = p.H[f * 64 + c_hi];
                w_hi = __fadd_rn(__fmul_rn(h1.x, h1.x), __fmul_rn(h1.y, h1.y));
            }
        }
        float m0 = lane == 0 ? 0.f : -INFINITY, m1 = -INFINITY;      // start in state 0
        uint2 keep = make_uint2(0u, 0u);
        for (int s = 0; s < n_sym; ++s) {
            const float2 *e = p.eq + (f * n_sym + s) * 48;
            const float2 e0 = e[lane];
            s_li[warp][2 * lane] = vit_input<DECISION>(w_lo, e0.x);
            s_li[warp][2 * lane + 1] = vit_input<DECISION>(w_lo, e0.y);
            if (lane < 16) {
                const float2 e1 = e[d_hi];
                s_li[warp][2 * d_hi] = vit_input<DECISION>(w_hi, e1.x);
                s_li[warp][2 * d_hi + 1] = vit_input<DECISION>(w_hi, e1.y);
            }
            __syncwarp();
#pragma unroll
            for (int m = 0; m < (N + 31) / 32; ++m) {
                const int j = lane + 32 * m;
                if (j >= N) break;
                float2 L;
                if (RATE == kCodeR12) {
                    L = make_float2(s_li[warp][ilv_pos(2 * j)], s_li[warp][ilv_pos(2 * j + 1)]);
                } else {                                                 // A0 B0 A1 B2 sent; stolen B1, A2 are erasures
                    const int g = j / 3, r = j - 3 * g, k = 4 * g;
                    L = r == 0 ? make_float2(s_li[warp][ilv_pos(k)], s_li[warp][ilv_pos(k + 1)])
                      : r == 1 ? make_float2(s_li[warp][ilv_pos(k + 2)], 0.f)
                               : make_float2(0.f, s_li[warp][ilv_pos(k + 3)]);
                }
                s_pair[warp][j] = L;
            }
            __syncwarp();
#pragma unroll 4
            for (int j = 0; j < N; ++j) {
                const int n = s * N + j;
                const float2 L = s_pair[warp][j];
                const float bm = __fadd_rn(sa * L.x, sb * L.y);
                const float a0 = __shfl_sync(0xffffffffu, m0, src), a1 = __shfl_sync(0xffffffffu, m1, src);
                const float b0 = __shfl_sync(0xffffffffu, m0, src + 1), b1 = __shfl_sync(0xffffffffu, m1, src + 1);
                const float me = lane < 16 ? a0 : a1, mo = lane < 16 ? b0 : b1;    // metrics of states 2 lane, 2 lane + 1
                const float c00 = __fadd_rn(me, bm), c01 = __fadd_rn(mo, -bm);      // -> state lane (input 0)
                const float c10 = __fadd_rn(me, -bm), c11 = __fadd_rn(mo, bm);      // -> state lane + 32 (input 1)
                const bool d0 = c01 > c00, d1 = c11 > c10;
                const float n0 = d0 ? c01 : c00, n1 = d1 ? c11 : c10;
                const uint32_t v0 = __ballot_sync(0xffffffffu, d0), v1 = __ballot_sync(0xffffffffu, d1);
                const float z = __shfl_sync(0xffffffffu, n0, 0);
                m0 = __fsub_rn(n0, z);
                m1 = __fsub_rn(n1, z);
                if ((n & 31) == lane) keep = make_uint2(v0, v1);
                if ((n & 31) == 31 || n == T - 1) {
                    if (lane <= (n & 31)) surv[(n & ~31) + lane] = keep;
                }
            }
            __syncwarp();
        }
        // traceback from state 0 (the tail terminates the trellis there)
        int state = 0;
        uint32_t f_err = 0;
        const int n_chunks = (T + 31) >> 5;
        for (int c = n_chunks - 1; c >= 0; --c) {
            const int n0 = c << 5;
            const uint2 mine = n0 + lane < T ? surv[n0 + lane] : make_uint2(0u, 0u);
            uint32_t word = 0;
#pragma unroll
            for (int k = 31; k >= 0; --k) {
                const uint32_t wx = __shfl_sync(0xffffffffu, mine.x, k), wy = __shfl_sync(0xffffffffu, mine.y, k);
                if (n0 + k < T) {
                    const uint32_t dec = ((state < 32 ? wx : wy) >> (state & 31)) & 1u;
                    word |= (uint32_t)(state >> 5) << k;
                    state = ((state << 1) & 63) | (int)dec;
                }
            }
            if (p.decoded != nullptr && lane == 0) p.decoded[f * n_words + c] = word;
            if (p.info != nullptr) {
                const int valid = k_info - n0;
                const uint32_t mask = valid >= 32 ? 0xffffffffu : valid <= 0 ? 0u : (1u << valid) - 1u;
                f_err += __popc((word ^ p.info[f * n_words + c]) & mask);
            }
        }
        if (p.decoded != nullptr && lane == 0)
            for (int c = n_chunks; c < n_words; ++c) p.decoded[f * n_words + c] = 0u;
        if (lane == 0) { a_err += f_err; a_ferr += f_err != 0; a_frames += 1; }
        __syncwarp();
    }
    if (p.counters == nullptr) return;
    if (lane == 0 && a_frames != 0) {
        ofdm_counters *o = p.counters;
        atomicAdd(reinterpret_cast<unsigned long long *>(&o->bit_errors), (unsigned long long)a_err);
        atomicAdd(reinterpret_cast<unsigned long long *>(&o->frames_in_error), (unsigned long long)a_ferr);
        atomicAdd(reinterpret_cast<unsigned long long *>(&o->frames), (unsigned long long)a_frames);
        atomicAdd(reinterpret_cast<unsigned long long *>(&o->bits), (unsigned long long)a_frames * (unsigned long long)k_info);
    }
}

}  // namespace ofdm
