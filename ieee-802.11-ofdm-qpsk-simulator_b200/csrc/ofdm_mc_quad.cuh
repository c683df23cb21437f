// ofdm_mc_quad.cuh -- k_mc_quad: the fused on-chip Monte-Carlo sweep of configs[3] (main()'s loop OFDM.c:1202-1222 with the
// payload bits and the noise drawn on chip) with one frame per 8-lane group.
//
// k_mc_philox (ofdm_chain.cuh) gives a warp one frame at a time: four transforms side by side per SNR point, then an exchange
// of 4 x 64 bins through shared memory.  Here a warp works on four consecutive frames, one per lane group, exactly as
// k_stream_quad (ofdm_stream.cuh) does for HBM-resident frames: per frame and SNR point the two noisy LTS halves are added in
// time and transformed once (three transforms instead of four), the estimate and the decisions stay in the registers of the
// lane that owns bins {u + 8j}, seven decision slots per symbol, rail errors and verdicts collected as sign bits.  The frame
// itself -- Philox payload bits, QPSK map, IFFT, cyclic prefix, power (OFDM.c:500-565, 637-643) -- is built once per frame by
// its lane group and its two symbol bodies stay in shared memory for all SNR points; nothing but the counters touches HBM.
//
// Streams, draws and their assignment to samples are those of k_mc_philox (DESIGN.md "Philox streams"): the sweep's result
// depends only on (seed, global frame index), not on which kernel, warp or lane group produced it.  kArithChecked = exact
// transmitter, power and noise scale, receiver speculated in fp32 with every decision verified and doubtful (frame, point)s
// replayed in the reference's arithmetic by the whole warp (frame_replay_exact): the totals of the all-exact kernel.  The error
// radii are those of k_stream_quad (halves added in time: 269 u S + 2 chan <= r_A + r_B).
#pragma once
#include "ofdm_stream.cuh"

namespace ofdm {

constexpr int kMcQuadWarps = 6;         // 2 blocks x 6 warps per SM: 168 registers (see k_stream_quad)

struct alignas(16) McQuadWarp {
    float2 tile[kWarpTile];             // transform transpose tiles (one per lane group); scratch of the exact replay
    float2 lts[2][kWin];                // scratch of the exact replay
    float2 body[4][2 * kWin + 8];       // the four frames' two symbol bodies in time (skewed windows; group pitch = 8 mod 16: half-warps hit distinct bank pairs)
    uint2 res[4][kMaxSnr];              // per frame and SNR point of the current quad: {packed rail errors, sum |e|^2}
    float sig[4][kMaxSnr];              // kArithChecked: the noise scale of every (frame, point)
    double terms[4][168];               // kArithChecked: |sample|^2 of the frame's 160 data samples in double, in frame order (:640)
};
inline size_t mc_quad_smem_bytes() { return sizeof(McQuadWarp) * kMcQuadWarps + 2 * kWin * sizeof(float2); }

// configs[4] fused the same way (fp32 arithmetic only: the verified multipath sweep is faster staged through HBM, DESIGN.md):
// per-frame random taps (Philox domain 2, as k_multipath<true>) applied by the frame's lane group to its own 320 samples, in
// k_multipath's operation order; the power is that of the faded frame; the faded LTS halves go to fwl, the faded symbol
// bodies replace the clean ones in place, last symbol first (a symbol's faded samples depend on nothing after it: n_taps <= 16).
struct alignas(16) McQuadWarpMp {
    float2 tile[kWarpTile];
    float2 body[4][2 * kWin + 8];       // clean, then faded symbol bodies
    float2 fwl[4][2 * kWin + 8];        // faded LTS halves
    float2 taps[4][kMaxTaps];
    float2 stage[4][96];                // 15 samples of history + the 80 clean samples (CP + body) of the symbol being faded, contiguous
    uint2 res[4][kMaxSnr];
};
inline size_t mc_quad_mp_smem_bytes() { return sizeof(McQuadWarpMp) * kMcQuadWarps + 160 * sizeof(float2); }
template <bool MP> struct McQuadSmem { using type = McQuadWarp; };
template <> struct McQuadSmem<true> { using type = McQuadWarpMp; };

// CH, the channel (DESIGN.md "Channels"; 0 = the reference's): kChComplex = circular complex noise, the Q-rail draws from
// domain 4 in the blocks of the I-rail ones; kChFixedSigma = the noise scale does not depend on the frame (Es/N0, Eb/N0): no
// frame power is measured and p.inv_sqrt_snr[i] holds point i's sigma itself.  Otherwise sigma = sqrt(P) * p.inv_sqrt_snr[i].
enum { kChComplex = 1, kChFixedSigma = 2 };

template <int ARITH, bool MP = false, int CH = 0>
__global__ void __launch_bounds__(kMcQuadWarps * 32, 2) k_mc_quad(McParams p)
{
    static_assert(ARITH == kArithFast || ARITH == kArithChecked, "the all-exact arithmetic runs in k_mc_philox");
    static_assert(!MP || ARITH == kArithFast, "the fused multipath variant is fp32 only");
    static_assert(CH == 0 || ARITH == kArithFast, "the fused channel variants are fp32 only (EXACT runs staged)");
    constexpr bool COMPLEX = (CH & kChComplex) != 0, FIXED = (CH & kChFixedSigma) != 0;
    constexpr bool CHECKED = ARITH == kArithChecked;
    constexpr int LEVEL = CHECKED ? 2 : 0;                        // fast: plain fp32 (statistical results, no EVM guard: as k_mc_philox)
    constexpr int WARPS = kMcQuadWarps;
    extern __shared__ __align__(128) unsigned char s_raw[];
    using WS = typename McQuadSmem<MP>::type;
    WS *ws_all = reinterpret_cast<WS *>(s_raw);
    float2 *s_ltsx = reinterpret_cast<float2 *>(s_raw + sizeof(WS) * WARPS);    // [2][kWin]: the LTS halves in time; MP: the whole 160-sample LTS slot
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, u = lane & 7;
    WS &ws = ws_all[warp];
    float2 *tile = ws.tile + grp * kGroupPitch;
    Tw<false> tw; tw.load(u);
    const QuadLane ql = make_quad_lane(u);
    // transmitter: natural bin of slot i of the lane's frequency grid -> data index / pilot / null (input index n <-> centred (n+32)%64)
    int dmap_tx[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) dmap_tx[i] = c_tab.bin_data[8 * slot_m<CHECKED>(i) + u];
    if constexpr (MP) { for (int i = threadIdx.x; i < 160; i += WARPS * 32) s_ltsx[i] = c_tab.lts_time[i]; }
    else { for (int i = threadIdx.x; i < 128; i += WARPS * 32) s_ltsx[(i >> 6) * kWin + (i & 63)] = c_tab.lts_time[32 + i]; }
    __syncthreads();

    const double q = (double)kQpsk;
    const float inv_ref2 = (float)(1.0 / (96.0 * (2.0 * q * q)));
    // Per-SNR totals live in registers: lane L owns SNR points L and L + 32 (n_snr <= 64); float EVM sums flushed every 16 quads
    uint32_t m_i[2] = {0, 0}, m_q[2] = {0, 0}, m_b[2] = {0, 0}, m_ferr[2] = {0, 0};
    float m_e2[2] = {0.f, 0.f}, m_evm[2] = {0.f, 0.f};
    double d_e2[2] = {0.0, 0.0}, d_evm[2] = {0.0, 0.0};
    uint32_t n_done = 0, n_quads = 0;

    const long n_quads_all = (p.n_frames + 3) >> 2;
    for (long qd = (long)blockIdx.x * WARPS + warp; qd < n_quads_all; qd += (long)gridDim.x * WARPS) {
        const long f = 4 * qd + grp;
        const bool active = f < p.n_frames;                       // idle groups of the batch's last quad compute along and book nothing
        const uint64_t fr = p.frame0 + (uint64_t)f;
        // ---- payload bits (Philox, one block per symbol) and Transmitter :500-565 for the two symbols
        const uint4 b0 = Philox::run(make_uint4((uint32_t)fr, (uint32_t)(fr >> 32), 0u, kDomainBits), p.seed, 0u);
        const uint4 b1 = Philox::run(make_uint4((uint32_t)fr, (uint32_t)(fr >> 32), 1u, kDomainBits), p.seed, 0u);
        float pw = 0.f;
#pragma unroll 1
        for (int s = 0; s < 2; ++s) {
            const uint32_t w0 = s ? b1.x : b0.x, w1 = s ? b1.y : b0.y, w2 = s ? b1.z : b0.z;
            float2 v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int d = dmap_tx[i];
                float2 x = make_float2(0.f, -0.f);
                if (d >= 0) { x = qpsk_point(bit_pair(w0, w1, w2, d)); x.y = -x.y; }
                else if (d == -2) x.x = 1.f;
                else if (d == -3) x.x = -1.f;
                v[i] = x;
            }
            if constexpr (CHECKED) {                              // the exact twiddles live only here: twice per frame
                Tw<true> twx; twx.load(u);
                fft64<true>(v, twx, tile, u);
            } else {
                fft64<false>(v, tw, tile, u);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int np = u + 8 * ((j + 4) & 7);               // fft_shift inside ifft's fft() -> 32-sample rotation (Q4)
                const float2 y = make_float2(v[j].x * 0.015625f, -v[j].y * 0.015625f);
                ws.body[grp][s * kWin + np] = y;
                const float e = fmaf(y.x, y.x, y.y * y.y);
                pw += np >= 48 ? 2.f * e : e;                       // the CP repeats samples 48..63 (:559-565)
            }
        }
        __syncwarp();
        float P = 0.f;
        if constexpr (MP) {
            // taps of this frame (k_multipath<true>): i.i.d. complex Gaussian, E|h_l|^2 = 1 / n_taps
            const int n_taps = p.n_taps;
            if (2 * u < n_taps) {
                const float scale = sqrtf(0.5f / (float)n_taps);
                float z[4];
                philox_normals4(p.seed, 0u, fr, (uint32_t)u, kDomainTaps, z);
                ws.taps[grp][2 * u] = make_float2(scale * z[0], scale * z[1]);
                if (2 * u + 1 < n_taps) ws.taps[grp][2 * u + 1] = make_float2(scale * z[2], scale * z[3]);
            }
            __syncwarp();
            // clean frame sample n: the LTS slot, then (CP + body) x 2 (:559-581)
            auto clean = [&](int n) -> float2 {
                if (n < 160) return s_ltsx[n];
                const int s = n >= 240 ? 1 : 0, k = n - 160 - 80 * s;
                return ws.body[grp][s * kWin + (k < 16 ? 48 + k : k - 16)];
            };
            // y[n] = sum_l h[l] x[n-l], descending l, separate multiplies and adds (k_multipath's order), on a contiguous run of
            // clean samples: x[0] = the sample at the output's own position
            auto fir = [&](const float2 *x, int l_max) -> float2 {
                float ar = 0.f, ai = 0.f;
                for (int l = l_max; l >= 0; --l) {
                    const float2 a = x[-l], b = ws.taps[grp][l];
                    ar = __fadd_rn(ar, __fsub_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)));
                    ai = __fadd_rn(ai, __fadd_rn(__fmul_rn(a.x, b.y), __fmul_rn(a.y, b.x)));
                }
                return make_float2(ar, ai);
            };
            float pm = 0.f;
            for (int n = u; n < 160; n += 8) {                      // the LTS slot: guard interval (power only), then the two halves
                const float2 y = fir(s_ltsx + n, n_taps - 1 < n ? n_taps - 1 : n);
                if constexpr (!FIXED) pm = fmaf(y.x, y.x, fmaf(y.y, y.y, pm));
                if (n >= 32) ws.fwl[grp][((n - 32) >> 6) * kWin + ((n - 32) & 63)] = y;
            }
            // symbol 1 first: its cyclic prefix still needs the clean tail of symbol 0 (the taps reach 15 samples back), while
            // symbol 0 depends on nothing after itself
#pragma unroll 1
            for (int s = 1; s >= 0; --s) {
                float2 *st = ws.stage[grp];
                for (int i = u; i < 95; i += 8) st[i] = clean(145 + 80 * s + i);
                __syncwarp();                                     // ... after which nobody reads the clean symbol any more
                // lane u: samples k = u + 8 m of the symbol; m < 2 is the CP (power only), the rest its own share of the body
#pragma unroll 1
                for (int m = 0; m < 10; ++m) {
                    const float2 y = fir(st + 15 + u + 8 * m, n_taps - 1);
                    if constexpr (!FIXED) pm = fmaf(y.x, y.x, fmaf(y.y, y.y, pm));
                    if (m >= 2) ws.body[grp][s * kWin + u + 8 * (m - 2)] = y;
                }
                __syncwarp();
            }
            pm += __shfl_xor_sync(0xffffffffu, pm, 1);
            pm += __shfl_xor_sync(0xffffffffu, pm, 2);
            pm += __shfl_xor_sync(0xffffffffu, pm, 4);
            P = pm / 320.f;
        } else if constexpr (CHECKED) {
            // OFDM.c:637-643 on the 320-sample frame: the LTS prefix is a constant, the 160 data samples follow in order.  The
            // terms are speculated as x^2 + y^2 in double by the group's eight lanes; lane 0 runs the sequential float chain over
            // them and takes glibc's hypot()^2 only where the running sum is within 16 double ulps of a float tie (power_step,
            // ofdm_kernels.cuh: bit-identical for every margin)
            for (int i = u; i < 160; i += 8) {
                const int s = i >= 80 ? 1 : 0, k = i - 80 * s;
                const float2 y = ws.body[grp][s * kWin + (k < 16 ? 48 + k : k - 16)];
                ws.terms[grp][i] = __fma_rn((double)y.x, (double)y.x, __dmul_rn((double)y.y, (double)y.y));
            }
            __syncwarp();
            float acc = 0.f;
            if (u == 0) {
                double pd = (double)c_tab.lts_power_prefix;
                for (int i = 0; i < 160; ++i) {
                    const double s = __dadd_rn(pd, ws.terms[grp][i]);
                    const uint32_t lo = (uint32_t)__double2loint(s), hi = (uint32_t)__double2hiint(s);
                    const int dist = (int)(lo & 0x1fffffffu) - 0x10000000;
                    if ((uint32_t)(dist < 0 ? -dist : dist) > 16u && s > 1e-30 && s < 1e30) {
                        const uint32_t lo2 = lo + 0x10000000u;                          // round to float: add half an ulp, clear 29 bits
                        pd = __hiloint2double((int)(hi + (lo2 < lo ? 1u : 0u)), (int)(lo2 & 0xe0000000u));
                    } else {                                                            // the reference's operations, OFDM.c:640-641
                        const int sy = i >= 80 ? 1 : 0, k = i - 80 * sy;
                        const float2 y = ws.body[grp][sy * kWin + (k < 16 ? 48 + k : k - 16)];
                        const double h = hypot_glibc((double)y.x, (double)y.y);
                        pd = (double)__double2float_rn(__dadd_rn(pd, __dmul_rn(h, h)));
                    }
                }
                acc = (float)pd;
            }
            P = __fdiv_rn(__shfl_sync(0xffffffffu, acc, lane & 24), 320.f);
            // exact noise scale sqrt((double)(P / snr)) (:647, :651) of every SNR point, rounded to float (= the correctly rounded
            // float square root, tests/test_sigma_rounding.py), spread over the group's lanes
            for (int si = u; si < p.n_snr; si += 8) ws.sig[grp][si] = __fsqrt_rn(__fdiv_rn(P, p.snr_lin[si]));
            __syncwarp();
        } else if constexpr (!FIXED) {
            pw += __shfl_xor_sync(0xffffffffu, pw, 1);
            pw += __shfl_xor_sync(0xffffffffu, pw, 2);
            pw += __shfl_xor_sync(0xffffffffu, pw, 4);
            P = (pw + c_tab.lts_power_sum) * (1.f / 320.f);
        }
        float sqrtP = 1.f;
        if constexpr (!FIXED) asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sqrtP) : "f"(P));
        const float chan = CHECKED ? p.radius_chan * sqrtP : 0.f;
        // the lane's payload words, bit a of every data bin with L < 0 flipped (quad_slot)
        const uint32_t fw[2][3] = {{b0.x ^ ql.flip0, b0.y ^ ql.flip1, b0.z ^ ql.flip2}, {b1.x ^ ql.flip0, b1.y ^ ql.flip1, b1.z ^ ql.flip2}};

        // ---- SNR loop OFDM.c:1202: channel :635 + receiver :1018-1165 on the frame held in shared memory.  The group sums of
        // a point (three shuffle steps) are finished one iteration late, on top of the next point's Philox rounds.
        uint32_t pk_pend = 0;
        float e2_pend = 0.f;
#pragma unroll 1
        for (int si = 0; si < p.n_snr; ++si) {
            {
                uint32_t pk = pk_pend; float e2 = e2_pend;
#pragma unroll
                for (int o = 1; o < 8; o <<= 1) { pk += __shfl_xor_sync(0xffffffffu, pk, o); e2 += __shfl_xor_sync(0xffffffffu, e2, o); }
                if (u == 0 && si > 0) ws.res[grp][si - 1] = make_uint2(pk, __float_as_uint(e2));
            }
            float sigma_f;
            if constexpr (CHECKED) sigma_f = ws.sig[grp][si]; else sigma_f = sqrtP * p.inv_sqrt_snr[si];
            const uint32_t stream = p.stream[si];
            // noisy samples of the window whose Philox blocks start at blk (v[m] = x[u + 8m] + sigma z, real rail only: SURVEY Q1;
            // kChComplex: + i sigma z' with z' the normal in the same slot of domain 4)
            auto window = [&](const float2 *src, int blk, float2 (&v)[8], float2 &n2) {
                float za[4], zb[4];
                philox_normals4(p.seed, stream, fr, (uint32_t)(blk + u), kDomainNoise, za);
                philox_normals4(p.seed, stream, fr, (uint32_t)(blk + u + 8), kDomainNoise, zb);
#pragma unroll
                for (int m = 0; m < 8; ++m) {
                    float2 smp = src[u + 8 * m];
                    smp.x = fmaf(sigma_f, m < 4 ? za[m] : zb[m - 4], smp.x);               // speculated channel (kChanRadius)
                    if (CHECKED) n2 = __ffma2_rn(smp, smp, n2);
                    v[m] = smp;
                }
                if constexpr (COMPLEX) {
                    philox_normals4(p.seed, stream, fr, (uint32_t)(blk + u), kDomainNoiseQ, za);
                    philox_normals4(p.seed, stream, fr, (uint32_t)(blk + u + 8), kDomainNoiseQ, zb);
#pragma unroll
                    for (int m = 0; m < 8; ++m) v[m].y = fmaf(sigma_f, m < 4 ? za[m] : zb[m - 4], v[m].y);
                }
            };
            // ---- Channel_Estimation :830-850: the two noisy halves added in time, one transform; G = A + B at bins u + 8j
            float2 G[8];
            float inv2[7], thr_a[7], thr_b[7];
            float rH2 = 0.f;
            bool doubt = false;
            {
                float2 b[8];
                float2 n2 = make_float2(0.f, 0.f);
                if constexpr (MP) { window(ws.fwl[grp], 8, G, n2); window(ws.fwl[grp] + kWin, 24, b, n2); }
                else { window(s_ltsx, 8, G, n2); window(s_ltsx + kWin, 24, b, n2); }
#pragma unroll
                for (int m = 0; m < 8; ++m) G[m] = cadd(G[m], b[m]);
                if (CHECKED) rH2 = window_radius(n2, p.radius_scale * 1.41421366f, 2.f * chan);
                fft64_fast(G, tw.t, tile, u);
                G[3] = u < 3 ? G[3] : G[4];
                const float den_min4 = (p.evm_guard * rH2) * (p.evm_guard * rH2);
#pragma unroll
                for (int t = 0; t < 7; ++t) {
                    const float2 Gt = t < 4 ? G[t] : G[t + 1];
                    const float den = fmaf(Gt.x, Gt.x, Gt.y * Gt.y);
                    if (CHECKED) {
                        const bool safe = den < 1.6e14f && den > den_min4;
                        doubt = doubt || (((ql.valid >> t) & 1u) && !safe);
                        const float hc = fabsf(Gt.x) + fabsf(Gt.y);
                        thr_a[t] = hc + rH2; thr_b[t] = fmaf(1.2e-7f, hc, rH2);
                    }
                    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv2[t]) : "f"(0.5f * den));
                }
            }
            uint32_t f_i = 0, f_q = 0, f_both = 0;
            float2 e2v = make_float2(0.f, 0.f);
            // (kArithChecked: not unrolled -- with both symbols inline the verified loop is 25 KB of code and the 12 warps of an SM,
            // each at its own place, stall on instruction fetch: ncu no_instruction 1.6 per issue, IPC 2.0, 17.0 instead of 15.3 ms;
            // the fp32 loop is 20 KB unrolled and runs 10 % faster that way)
#pragma unroll (CHECKED ? 1 : 2)
            for (int s = 0; s < 2; ++s) {
                float2 v[8];
                float2 n2 = make_float2(0.f, 0.f);
                window(ws.body[grp] + s * kWin, 44 + 20 * s, v, n2);
                float rF = 0.f;
                if (CHECKED) rF = window_radius(n2, p.radius_scale, chan);
                fft64_fast(v, tw.t, tile, u);
                const uint32_t w0 = s ? fw[1][0] : fw[0][0], w1 = s ? fw[1][1] : fw[0][1], w2 = s ? fw[1][2] : fw[0][2];
                const uint32_t word_a = u < 2 ? w1 : w2, word_b = u < 3 ? w2 : w0, word_c = u == 7 ? w1 : w0;     // see k_stream_quad
                uint32_t acc_i = 0, acc_q = 0, acc_s = 0;
#pragma unroll
                for (int t = 0; t < 7; ++t) {
                    const float2 F = t < 3 ? v[t] : (t == 3 ? (u < 3 ? v[3] : v[4]) : v[t + 1]);
                    const float2 Gt = t < 4 ? G[t] : G[t + 1];
                    const uint32_t w = t == 0 ? w1 : t == 1 ? word_a : t == 2 ? w2 : t == 3 ? word_b : t == 4 ? w0 : t == 5 ? word_c : w1;
                    const uint32_t tb = __funnelshift_l(0u, w, (t < 4 ? ql.sh_lo : ql.sh_hi) >> (5 * (t & 3)));
                    quad_slot<LEVEL>(F, Gt, inv2[t], tb, (ql.valid >> t) & 1u, rF, thr_a[t], thr_b[t], acc_i, acc_q, acc_s, e2v);
                }
                if (CHECKED) doubt = doubt || (acc_s & ql.valid_rev) != ql.valid_rev;
                acc_i &= ql.valid_rev; acc_q &= ql.valid_rev;
                f_i += __popc(acc_i); f_q += __popc(acc_q); f_both += __popc(acc_i & acc_q);
            }
            uint32_t pk = f_i | (f_q << 8) | (f_both << 16);      // per lane at most 14 of each
            float e2 = e2v.x + e2v.y;
            if constexpr (CHECKED) {
                uint32_t dm = __ballot_sync(0xffffffffu, doubt && active);
                while (dm != 0u) {                                // warp-uniform: the whole warp replays one (frame, point) at a time
                    const int g = (__ffs((int)dm) - 1) >> 3;
                    dm &= ~(0xFFu << (8 * g));
                    const float Pg = __shfl_sync(0xffffffffu, P, 8 * g);
                    const double sigma_d = __dsqrt_rn((double)__fdiv_rn(Pg, p.snr_lin[si]));
                    const McFrame fr = {grp < 2 ? s_ltsx + grp * kWin : ws.body[g] + (grp - 2) * kWin};
                    const ReplayTotals rr = frame_replay_exact<kNoisePhilox>(fr, sigma_d, p.seed, stream, p.frame0 + (uint64_t)(4 * qd + g), ws.tile, &ws.lts[0][0], p.replayed);
                    const uint32_t tpk = __reduce_add_sync(0xffffffffu, rr.packed());
                    float te2 = rr.e2;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) te2 += __shfl_xor_sync(0xffffffffu, te2, o);
                    if (grp == g) { pk = u == 0 ? tpk : 0u; e2 = u == 0 ? te2 : 0.f; }
                }
            }
            pk_pend = pk; e2_pend = e2;
        }
        {
            uint32_t pk = pk_pend; float e2 = e2_pend;
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) { pk += __shfl_xor_sync(0xffffffffu, pk, o); e2 += __shfl_xor_sync(0xffffffffu, e2, o); }
            if (u == 0) ws.res[grp][p.n_snr - 1] = make_uint2(pk, __float_as_uint(e2));
        }
        __syncwarp();
        // the lane that owns an SNR point books the quad's four frames for it
        const int n_act = p.n_frames - 4 * qd < 4 ? (int)(p.n_frames - 4 * qd) : 4;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (h == 1 && p.n_snr <= 32) break;
            const bool mine = lane + 32 * h < p.n_snr;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const uint2 rr = ws.res[g][lane + 32 * h];
                const bool take = mine && g < n_act;
                const uint32_t pkh = take ? rr.x : 0u;
                const float e2h = take ? __uint_as_float(rr.y) : 0.f;
                float evm;
                asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(evm) : "f"(e2h * inv_ref2));                // :1124
                m_i[h] += pkh & 0xFFu; m_q[h] += (pkh >> 8) & 0xFFu; m_b[h] += pkh >> 16; m_ferr[h] += pkh != 0u;
                m_e2[h] += e2h; m_evm[h] += evm;
            }
        }
        __syncwarp();
        n_done += (uint32_t)n_act;
        if ((++n_quads & 15u) == 0u) {
#pragma unroll
            for (int h = 0; h < 2; ++h) { d_e2[h] += (double)m_e2[h]; d_evm[h] += (double)m_evm[h]; m_e2[h] = 0.f; m_evm[h] = 0.f; }
        }
    }
    if (n_done == 0) return;
    const double ref2_frame = 96.0 * (2.0 * q * q);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int si = lane + 32 * h;
        if (si >= p.n_snr) continue;
        ofdm_counters *o = p.counters + si;
        const unsigned long long ti = m_i[h], tq = m_q[h], tb = m_b[h];
        atomicAdd(reinterpret_cast<unsigned long long *>(&o->bit_errors), ti + 2ull * tq - 2ull * tb);     // map of :423-430
        atomicAdd(reinterpret_cast<unsigned long long *>(&o->rail_errors), ti + tq);
        atomicAdd(reinterpret_cast<unsigned long long *>(&o->frames_in_error), (unsigned long long)m_ferr[h]);
        atomicAdd(reinterpret_cast<unsigned long long *>(&o->frames), (unsigned long long)n_done);
        atomicAdd(reinterpret_cast<unsigned long long *>(&o->bits), 192ull * n_done);
        atomicAdd(&o->sum_err2, d_e2[h] + (double)m_e2[h]);
        atomicAdd(&o->sum_ref2, ref2_frame * (double)n_done);
        atomicAdd(&o->sum_evm_lin, d_evm[h] + (double)m_evm[h]);
    }
}

}  // namespace ofdm
