// ofdm_stream.cuh -- k_stream_quad: the streaming channel + receiver (OFDM.c:635-655, 1018-1165) for HBM-resident frames of
// any length, one frame per 8-lane group.
//
// k_stream_rx2 / k_stream_rxn (ofdm_chain.cuh) give a warp one frame at a time: its four lane groups transform the two LTS
// halves and two symbol bodies side by side, and the results have to change hands afterwards (the groups publish 4 x 64 bins
// to shared memory, the lanes pick up their items).  Those kernels are bound by shared-memory bandwidth (DESIGN 5.2:
// ~101 wavefronts per frame against the 150 cycles an SM spends on it).  Here each lane group owns a whole FRAME and a warp
// works on four consecutive frames:
//   * the group adds the two received LTS halves in time (the transform is linear: FFT(a) + FFT(b) = FFT(a + b)) and
//     transforms the sum once -- three transforms per two-symbol frame instead of four;
//   * the channel estimate G = A + B stays in the registers of the lane that owns bins {u + 8j}, and that same lane receives
//     the same bins of every data symbol: equalise / slice / demod / EVM / BER need no exchange at all;
//   * what is left per frame in shared memory is one trip through the TMA ring per window and one 8x8 transpose per
//     transform: 56 wavefronts for a two-symbol frame (+ 24 with injected draws; ncu counts 49 / 61 against 112 / 120), and a
//     quarter fewer instructions (247 instead of 328 per frame for the fp32 receiver, 376 instead of 479 verified with draws).
// The price is lane utilisation in the decision stage: a lane's eight bins hold five to seven data bins (null / pilot bins
// idle); bins 24+u and 32+u are complementary (three and two data bins) and share one slot, so 7 slots x 8 lanes serve the
// 48 data bins of a symbol (86 %).
//
// TMA ring: per warp DEPTH slots, a slot = ONE 64-sample window of the warp's four frames (4 x 512 B of IQ, + 4 x 256 B of
// draws), filled by cp.async.bulk copies that one elected lane issues, completion on the slot's mbarrier.  The units of a
// quad of frames are consumed in order -- LTS half 1, LTS half 2, symbol 0, 1, ... -- and a slot is refilled with the unit
// DEPTH positions ahead as soon as the lanes have pulled their samples into registers.
//
// Arithmetic: kArithFast (fp32, EVM guard only) and kArithChecked (fp32 speculation, every rail decision verified, doubtful
// frames replayed in the reference's arithmetic) exactly as in ofdm_chain.cuh; the all-exact kernels stay k_stream_rx2 / rxn.
// Error radius of the channel estimate with the halves added in time (u = 2^-24, S = |a'|_2 + |b'|_2 the norms of the noisy
// halves, see the derivation at kRadius):
//   reference  fl(FFT_ref(a') + FFT_ref(b')):  97 u S (its butterflies) + 16 u S (rounding of the sum, |A + B| <= 8 S)
//   this path  FFT_fp32(fl(a~ + b~)):  8 u S (rounding of the sum in time, carried through the transform) + 116 u S (fp32
//              transform) + 32 u S + 2 x 16 u |x|_2 (speculated channel: a~ vs a', the kChanRadius term)
//   => |G~ - G_ref| <= 269 u S + 2 chan <= r_A + r_B with r = kRadius |window|_2 + chan, kRadius = 320 u: the same
//   expression the four-transform kernels use for 2 r_H.  F is unchanged (97 + 116 + 32 = 245 u).
#pragma once
#include "ofdm_chain.cuh"

namespace ofdm {

template <bool WITH_DRAWS> struct alignas(16) QuadSlot {        // bulk-copy destinations must be 16-byte aligned
    float2 x[4][kWin];              // one window of the warp's four frames (skewed pitch: half-warps hit distinct bank pairs)
    float g[4][kWin];               // the matching draws
};
template <> struct alignas(16) QuadSlot<false> { float2 x[4][kWin]; };

#ifndef OFDM_QUAD_DEPTH
#define OFDM_QUAD_DEPTH 4               // A/B knobs (tools/ab.sh): ring slots per warp without / with injected draws
#endif
#ifndef OFDM_QUAD_DEPTH_DRAWS
#define OFDM_QUAD_DEPTH_DRAWS 4
#endif
template <int NOISE> __host__ __device__ constexpr int quad_depth() { return NOISE == kNoiseInject ? OFDM_QUAD_DEPTH_DRAWS : OFDM_QUAD_DEPTH; }

template <int NOISE> struct alignas(16) QuadWarp {
    float2 tile[kWarpTile];         // transform transpose tiles (one per lane group); scratch of the exact replay
    float2 lts[2][kWin];            // scratch of the exact replay
    QuadSlot<NOISE == kNoiseInject> slot[quad_depth<NOISE>()];
    uint64_t bar[quad_depth<NOISE>()];
};
// Block shape: the kernel wants ~170 registers to keep a frame's estimate, a symbol's bins and the per-lane constants
// resident; 2 blocks x 6 warps per SM give it 168 (12 warps per SM; latency is covered by the TMA ring, not by occupancy).
// 8 warps per block (128 registers, 16 warps per SM) is kept as an A/B knob ("stream_warps").
template <int NOISE> inline size_t quad_smem_bytes(int warps) { return sizeof(QuadWarp<NOISE>) * warps; }

// Per-lane constants of the seven decision slots: slot t holds bin u + 8 j with j = t (t < 3), 3 or 4 (t = 3: lanes 0..2 own the
// data bins 24..26, lanes 6, 7 the data bins 38, 39), t + 1 (t > 3).  The payload word of a slot's bit pair is fixed per slot
// up to three lane-dependent choices (word_a / word_b / word_c below), its position inside the word is a per-lane constant.
struct QuadLane {
    uint32_t flip0, flip1, flip2;   // per payload word: bit 2d set for each of the lane's data bins d with L < 0 (see quad_slot)
    uint32_t sh_lo, sh_hi;          // 5-bit fields: 30 - 2 (d & 15) of slots 0..3 and 4..6
    uint32_t valid;                 // bit t: the slot's bin is a data bin
    uint32_t valid_rev;             // the same, bit 6 - t (the order in which the slots' sign bits are collected)
};
__device__ __forceinline__ QuadLane make_quad_lane(int u)
{
    QuadLane c = {0u, 0u, 0u, 0u, 0u, 0u, 0u};
#pragma unroll
    for (int t = 0; t < 7; ++t) {
        const int j = t < 3 ? t : (t == 3 ? (u < 3 ? 3 : 4) : t + 1);
        const int bin = u + 8 * j;
        const int d = c_tab.bin_data[bin];
        const uint32_t sh = 30u - 2u * (uint32_t)(d & 15);
        if (t < 4) c.sh_lo |= sh << (5 * t); else c.sh_hi |= sh << (5 * (t - 4));
        if (d >= 0) {
            c.valid |= 1u << t;
            c.valid_rev |= 1u << (6 - t);
            const uint32_t bit = c_tab.bin_lts[bin] < 0 ? 1u << (2 * (d & 15)) : 0u;
            c.flip0 |= d < 16 ? bit : 0u; c.flip1 |= (d >= 16 && d < 32) ? bit : 0u; c.flip2 |= d >= 32 ? bit : 0u;
        }
    }
    return c;
}

// One data bin of one symbol: equalise :1050, slicer :860-868, demod :883-902, BER :1158 and the EVM term :1114, speculated in
// fp32 (the arithmetic and tests of process_bin_spec, ofdm_chain.cuh).  Per frame the caller has formed G = A + B (unscaled
// estimate, H = 0.5 L G :848), inv2 = 2 / |G|^2 and checked |G|^2 against the EVM guard and the magnitude bound.
// tb = payload word shifted so that bit 31 = b, bit 30 = a of the bin's pair, bit a already flipped where L < 0.  With
// S = F conj(G) the equalised point is E = L S inv2; multiplying Re S by the sign of the transmitted I rail (a ^ b,
// QPSK_Modulator :423-430) and of L, Im S by those of the Q rail (a) and L, makes the bin look as if (+1, +1)/sqrt(2) had been
// sent through L = +1: a rail error is the sign bit of S, the error vector is S inv2 - (h, h).  The sign bits are collected into
// acc_i / acc_q (one funnel shift each), counted once per symbol.
__device__ __forceinline__ float xor_sign(float x, uint32_t bits)
{
    return __uint_as_float(__float_as_uint(x) ^ (bits & 0x80000000u));
}
// thr_a, thr_b (kArithChecked): the parts of the decision threshold that do not depend on the symbol, per frame and slot --
// |speculated - reference numerator| <= rF |G|_1 + rH2 |F|_1 + rF rH2, + 2^-23 |F|_1 |G|_1 for the fp32 evaluation, i.e.
// thr = rF thr_a + |F|_1 thr_b with thr_a = |G|_1 + rH2, thr_b = rH2 + 1.2e-7 |G|_1.
// The verdict of a slot joins acc_s the same way: the sign bit of thr - min(|Re S|, |Im S|) is set exactly when the smaller
// rail exceeds the threshold (an infinite or NaN threshold -- window energies out of range, non-finite samples -- gives +Inf
// or the canonical NaN 0x7fffffff PTX arithmetic returns: sign bit clear, not trusted).
template <int LEVEL>
__device__ __forceinline__ void quad_slot(float2 F, float2 G, float inv2, uint32_t tb, bool valid, float rF, float thr_a, float thr_b,
                                          uint32_t &acc_i, uint32_t &acc_q, uint32_t &acc_s, float2 &e2)
{
    const uint32_t ta = tb << 1;
    const float2 pt = __fmul2_rn(make_float2(G.y, G.y), make_float2(F.y, F.x));
    float2 S = __ffma2_rn(make_float2(G.x, G.x), F, make_float2(pt.x, -pt.y));       // (fma(a, c, b d), fma(b, c, -(a d)))
    S.x = xor_sign(S.x, ta ^ tb);
    S.y = xor_sign(S.y, ta);
    if (LEVEL >= 2) {
        // trusted only if the smaller rail of the numerator exceeds the threshold, which carries an absolute 2e-30 (the reference's
        // numerator is then at least 2e-30 in magnitude and its float quotient keeps the sign: |G|^2 < 1.6e14; where the addend is
        // lost to rounding, thr > 3e-23 and one float step above it is already more than 2e-30); NaN / Inf fail the comparison
        const float fa = fabsf(F.x) + fabsf(F.y);
        const float thr = fmaf(fa, thr_b, fmaf(rF, thr_a, 2e-30f));
        acc_s = __funnelshift_l(__float_as_uint(thr - fminf(fabsf(S.x), fabsf(S.y))), acc_s, 1);
    }
    const float2 D = __ffma2_rn(S, make_float2(inv2, inv2), make_float2(-kQpsk, -kQpsk));
    if (valid) e2 = __ffma2_rn(D, D, e2);
    acc_i = __funnelshift_l(__float_as_uint(S.x), acc_i, 1);
    acc_q = __funnelshift_l(__float_as_uint(S.y), acc_q, 1);
}

// NSYM2 (the default frame shape, two data symbols): a quad has four units and the ring four slots, so unit w of every quad
// travels through slot w, one quad ahead of its use -- slot, barrier, window offset and frame pitch are compile-time constants
// at each of the four places a unit is taken, and a refill is an elected lane adding immediates to the next quad's base
// address (23 instead of 42 instructions per refill; the refill path was 23 % of the general kernel's stall samples).
template <int W> struct UnitIndex { static constexpr int value = W; };

template <int ARITH, int NOISE, int WARPS, bool NSYM2 = false>
__global__ void __launch_bounds__(WARPS * 32, 2) k_stream_quad(RxParams p)
{
    static_assert(ARITH == kArithFast || ARITH == kArithChecked, "the all-exact arithmetic runs in k_stream_rx2 / k_stream_rxn");
    constexpr int LEVEL = ARITH == kArithChecked ? 2 : 1;
    constexpr int DEPTH = quad_depth<NOISE>();
    constexpr bool DRAWS = NOISE == kNoiseInject;
    static_assert(!NSYM2 || DEPTH == 4, "NSYM2: one ring slot per unit of a quad");
    extern __shared__ __align__(128) unsigned char s_raw[];
    __shared__ unsigned long long s_cnt[WARPS][4];
    __shared__ double s_sum[WARPS][2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, u = lane & 7;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);                  // same value, provably warp-uniform
    using QW = QuadWarp<NOISE>;
    using QS = QuadSlot<DRAWS>;
    QW &ws = reinterpret_cast<QW *>(s_raw)[warp];
    QW &ws_u = reinterpret_cast<QW *>(s_raw)[warp_u];
    float2 *tile = ws.tile + grp * kGroupPitch;
    Tw<false> tw; tw.load(u);
    const QuadLane ql = make_quad_lane(u);
    const int n_sym = NSYM2 ? 2 : p.n_sym, len = 160 + 80 * n_sym;
    const long n_quads = (p.n_frames + 3) >> 2;
    const long wstride = (long)gridDim.x * WARPS;
    const long q_first = (long)blockIdx.x * WARPS + warp_u;
    const int my_quads = q_first < n_quads ? (int)((n_quads - q_first + wstride - 1) / wstride) : 0;
    const double q = (double)kQpsk;
    const double ref2_frame = 48.0 * n_sym * (2.0 * q * q);     // sum |tx|^2 over the frame's data bins
    const float inv_ref2 = (float)(1.0 / ref2_frame);

    // A refill = one expect_tx + one bulk copy per frame of the quad (two with draws), issued by one elected lane; all
    // operands derive from warp-uniform values and stay on the uniform datapath (UBLKCP).  The producer keeps the address of
    // the next unit's window in the quad's first frame and steps it from unit to unit.
    const uint32_t slot0 = tma::saddr(&ws_u.slot[0]);
    const uint32_t bar0 = tma::saddr(&ws_u.bar[0]);
    const long len8 = (long)len * 8, len4 = (long)len * 4;
    const long quad_step = 4 * wstride - 1;                       // frames from the last unit of a quad to the first unit of the warp's next quad, less one
    const char *ix = reinterpret_cast<const char *>(p.in) + 4 * len8 * q_first + 32 * 8;       // Channel_Estimation :837
    const char *ig = reinterpret_cast<const char *>(p.g) + 4 * len4 * q_first + 32 * 4;
    long i_left = p.n_frames - 4 * q_first;                       // frames from that quad's first frame to the end of the batch
    int i_togo = n_sym + 1;                                       // units of that quad after the next one
    auto issue_next = [&](int s) {
        if (i_left > 0) {
            if (tma::elect_one()) {
                const uint32_t bar = bar0 + 8u * (uint32_t)s;
                const uint32_t dst = slot0 + (uint32_t)s * (uint32_t)sizeof(QS);
                const uint32_t gd = dst + 4 * kWin * 8;
                if (i_left >= 4) {
                    tma::expect_tx_addr(bar, DRAWS ? 4 * 768u : 4 * 512u);
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        tma::bulk_addr(dst + (uint32_t)g * kWin * 8, ix + g * len8, 512, bar);
                        if (DRAWS) tma::bulk_addr(gd + (uint32_t)g * kWin * 4, ig + g * len4, 256, bar);
                    }
                } else {                                          // the last quad of the batch, when it is not whole
                    const int n_act = (int)i_left;
                    tma::expect_tx_addr(bar, (uint32_t)n_act * (DRAWS ? 768u : 512u));
                    for (int g = 0; g < n_act; ++g) {
                        tma::bulk_addr(dst + (uint32_t)g * kWin * 8, ix + g * len8, 512, bar);
                        if (DRAWS) tma::bulk_addr(gd + (uint32_t)g * kWin * 4, ig + g * len4, 256, bar);
                    }
                }
            }
            // next unit: LTS half 2 is 64 samples on (:838), every other unit 80 (:1028); after the last symbol the first
            // half of the warp's next quad: the rest of this frame (64 samples), the frames in between, and 32 samples
            if (i_togo == 0) {
                ix += quad_step * len8 + (64 + 32) * 8; ig += quad_step * len4 + (64 + 32) * 4;
                i_left -= 4 * wstride; i_togo = n_sym + 1;
            } else {
                const int step = i_togo == n_sym + 1 ? 64 : 80;
                ix += step * 8; ig += step * 4;
                --i_togo;
            }
        }
    };
    // NSYM2: the quad whose units the next refills fetch (the one after the quad being consumed): base addresses, frames in it
    const char *nx = reinterpret_cast<const char *>(p.in) + 4 * len8 * q_first;
    const char *ng = reinterpret_cast<const char *>(p.g) + 4 * len4 * q_first;
    int n_next = 0;
    auto refill = [&](auto Wc) {
        constexpr int W = decltype(Wc)::value;
        constexpr int n0 = W == 0 ? 32 : (W == 1 ? 96 : (W == 2 ? 176 : 256));                // :837, :838, :1028
        constexpr long kLen8 = 320 * 8, kLen4 = 320 * 4;
        if (n_next > 0) {
            if (tma::elect_one()) {
                const uint32_t bar = bar0 + 8u * W;
                const uint32_t dst = slot0 + (uint32_t)W * (uint32_t)sizeof(QS);
                const uint32_t gd = dst + 4 * kWin * 8;
                tma::expect_tx_addr(bar, (uint32_t)n_next * (DRAWS ? 768u : 512u));
                if (n_next == 4) {
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        tma::bulk_addr(dst + (uint32_t)g * kWin * 8, nx + (n0 * 8 + g * kLen8), 512, bar);
                        if (DRAWS) tma::bulk_addr(gd + (uint32_t)g * kWin * 4, ng + (n0 * 4 + g * kLen4), 256, bar);
                    }
                } else {                                          // the last quad of the batch, when it is not whole
                    for (int g = 0; g < n_next; ++g) {
                        tma::bulk_addr(dst + (uint32_t)g * kWin * 8, nx + (n0 * 8 + g * kLen8), 512, bar);
                        if (DRAWS) tma::bulk_addr(gd + (uint32_t)g * kWin * 4, ng + (n0 * 4 + g * kLen4), 256, bar);
                    }
                }
            }
        }
    };
    if (lane == 0) {
        for (int s = 0; s < DEPTH; ++s) tma::mbar_init(&ws.bar[s], 1);
        tma::fence_mbar_init();
    }
    __syncwarp();
    if constexpr (NSYM2) {
        const long left = p.n_frames - 4 * q_first;
        n_next = left <= 0 ? 0 : (left < 4 ? (int)left : 4);      // the warp's first quad
        refill(UnitIndex<0>{}); refill(UnitIndex<1>{}); refill(UnitIndex<2>{}); refill(UnitIndex<3>{});
    } else {
#pragma unroll 1
        for (int s = 0; s < DEPTH; ++s) issue_next(s);
    }

    int cs = 0;                                                   // ring position of the unit being consumed
    uint32_t cph = 0;
    // pull the lane's eight samples of the current unit (v[m] = x[u + 8m]), add the noise, release the slot
    auto take = [&](auto Wc, float2 (&v)[8], float2 &n2, float sigma_f, long f, int n0) {
        constexpr int W = decltype(Wc)::value;                    // NSYM2: the unit's place in the quad = its ring slot
        [[maybe_unused]] float z[8];
        if constexpr (NOISE == kNoisePhilox) {                    // Philox noise of the window that starts at sample n0
            const int blk = window_block_base(n0) + u;
            float za[4], zb[4];
            philox_normals4(p.seed, p.stream, p.frame0 + (uint64_t)f, (uint32_t)blk, kDomainNoise, za);
            philox_normals4(p.seed, p.stream, p.frame0 + (uint64_t)f, (uint32_t)(blk + 8), kDomainNoise, zb);
#pragma unroll
            for (int m = 0; m < 4; ++m) { z[m] = za[m]; z[4 + m] = zb[m]; }
        }
        tma::wait_addr(bar0 + 8u * (uint32_t)(NSYM2 ? W : cs), cph);
        const QS &sl = ws.slot[NSYM2 ? W : cs];
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            float2 smp = sl.x[grp][u + 8 * m];
            if constexpr (DRAWS) smp.x = fmaf(sigma_f, sl.g[grp][u + 8 * m], smp.x);      // speculated channel (kChanRadius)
            if constexpr (NOISE == kNoisePhilox) smp.x = fmaf(sigma_f, z[m], smp.x);
            n2 = __ffma2_rn(smp, smp, n2);
            v[m] = smp;
        }
        __syncwarp();                                             // every lane has its samples: the slot can be refilled
        if constexpr (NSYM2) {
            refill(Wc);
            if (W == 3) cph ^= 1u;
        } else {
            issue_next(cs);
            if (++cs == DEPTH) { cs = 0; cph ^= 1u; }
        }
    };

    uint32_t a_i = 0, a_q = 0, a_both = 0, a_ferr = 0, a_frames = 0;     // per lane
    double a_e2 = 0.0, a_evm = 0.0;                                      // lanes u == 0: their group's frames
    for (int jc = 0; jc < my_quads; jc += 8) {
        // lane l prepares the noise scale sqrt((double)(P / snr_lin)) (:647, :651) of frame (l & 3) of the chunk's quad l >> 2
        float sig_mine = 0.f;
        if (NOISE != kNoiseNone) {
            const int jl = jc + (lane >> 2);
            const long fl = 4 * (q_first + (long)jl * wstride) + (lane & 3);
            if (jl < my_quads && fl < p.n_frames) sig_mine = (float)__dsqrt_rn((double)__fdiv_rn(p.power[fl], p.snr_lin));
        }
        float c_e2 = 0.f, c_evm = 0.f;
#pragma unroll 1
        for (int kk = 0; kk < 8; ++kk) {
            const int jq = jc + kk;
            if (jq >= my_quads) break;
            const long f0 = 4 * (q_first + (long)jq * wstride);
            if constexpr (NSYM2) {                                // this quad's refills fetch the warp's next quad
                const long f0n = f0 + 4 * wstride, left = p.n_frames - f0n;
                nx = reinterpret_cast<const char *>(p.in) + f0n * (320 * 8);
                ng = reinterpret_cast<const char *>(p.g) + f0n * (320 * 4);
                n_next = left <= 0 ? 0 : (left < 4 ? (int)left : 4);
            }
            const long f = f0 + grp;
            const bool active = f < p.n_frames;                   // only the batch's last quad can have idle groups: they compute along on stale samples
            const float sigma_f = NOISE != kNoiseNone ? __shfl_sync(0xffffffffu, sig_mine, 4 * kk + grp) : 0.f;
            const float chan = NOISE != kNoiseNone ? p.radius_chan * sigma_f : 0.f;
            // payload words of the frame's first symbol, fetched a whole unit ahead of their use (every later symbol's likewise)
            const uint32_t *wb = p.tx_bits + (active ? f : 0) * ((long)n_sym * 3);
            uint32_t nw0 = __ldg(wb), nw1 = __ldg(wb + 1), nw2 = __ldg(wb + 2);
            // ---- Channel_Estimation :830-850: the two halves added in time, one transform; G = A + B (unscaled) at bins u + 8j
            float2 G[8];
            float inv2[7], thr_a[7], thr_b[7];
            float rH2;
            bool doubt = false;
            {
                float2 b[8];
                float2 n2 = make_float2(0.f, 0.f);
                take(UnitIndex<0>{}, G, n2, sigma_f, f, 32);
                take(UnitIndex<1>{}, b, n2, sigma_f, f, 96);
#pragma unroll
                for (int m = 0; m < 8; ++m) G[m] = cadd(G[m], b[m]);
                // 2 r_H = kRadius (|a|_2 + |b|_2) + 2 chan, and |a|_2 + |b|_2 <= sqrt(2) sqrt(|a|_2^2 + |b|_2^2)
                rH2 = window_radius(n2, p.radius_scale * 1.41421366f, 2.f * chan);
                fft64_fast(G, tw.t, tile, u);
                G[3] = u < 3 ? G[3] : G[4];                       // slot 3; G[4] is dead from here on
                // reference |H|^2 < 1e14 (the float quotient keeps its sign) and the EVM guard |H| >= evm_guard radii
                const float den_min4 = (p.evm_guard * rH2) * (p.evm_guard * rH2);
#pragma unroll
                for (int t = 0; t < 7; ++t) {
                    const float2 Gt = t < 4 ? G[t] : G[t + 1];
                    const float den = fmaf(Gt.x, Gt.x, Gt.y * Gt.y);
                    const bool safe = den < 1.6e14f && den > den_min4;
                    doubt = doubt || (((ql.valid >> t) & 1u) && !safe);
                    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv2[t]) : "f"(0.5f * den));
                    if (LEVEL >= 2) {
                        const float hc = fabsf(Gt.x) + fabsf(Gt.y);
                        thr_a[t] = hc + rH2; thr_b[t] = fmaf(1.2e-7f, hc, rH2);
                    }
                }
            }
            uint32_t f_i = 0, f_q = 0, f_both = 0;
            float2 e2v = make_float2(0.f, 0.f);
            // ---- data symbols :1020-1069 against the estimate in registers
            auto symbol = [&](auto Wc, int s) {
                const uint32_t w0 = nw0 ^ ql.flip0, w1 = nw1 ^ ql.flip1, w2 = nw2 ^ ql.flip2;
                if (s + 1 < n_sym) { wb += 3; nw0 = __ldg(wb); nw1 = __ldg(wb + 1); nw2 = __ldg(wb + 2); }
                float2 v[8];
                float2 n2 = make_float2(0.f, 0.f);
                take(Wc, v, n2, sigma_f, f, 176 + 80 * s);
                float rF = 0.f;
                if (LEVEL >= 2) rF = window_radius(n2, p.radius_scale, chan);
                fft64_fast(v, tw.t, tile, u);
                // payload word of each slot: bins 1..6 -> d 24..29, 8..20 -> 30..42, 22..26 -> 43..47, 38..42 -> 0..4, 44..56 -> 5..17, 58..63 -> 18..23
                const uint32_t word_a = u < 2 ? w1 : w2;          // slot 1: bins 8 + u
                const uint32_t word_b = u < 3 ? w2 : w0;          // slot 3: bins 24 + u (u < 3) / 32 + u (u > 5)
                const uint32_t word_c = u == 7 ? w1 : w0;         // slot 5: bins 48 + u
                uint32_t acc_i = 0, acc_q = 0, acc_s = 0;
#pragma unroll
                for (int t = 0; t < 7; ++t) {
                    const float2 F = t < 3 ? v[t] : (t == 3 ? (u < 3 ? v[3] : v[4]) : v[t + 1]);
                    const float2 Gt = t < 4 ? G[t] : G[t + 1];
                    const uint32_t w = t == 0 ? w1 : t == 1 ? word_a : t == 2 ? w2 : t == 3 ? word_b : t == 4 ? w0 : t == 5 ? word_c : w1;
                    const uint32_t tb = __funnelshift_l(0u, w, (t < 4 ? ql.sh_lo : ql.sh_hi) >> (5 * (t & 3)));      // w << (field & 31)
                    quad_slot<LEVEL>(F, Gt, inv2[t], tb, (ql.valid >> t) & 1u, rF, thr_a[t], thr_b[t], acc_i, acc_q, acc_s, e2v);
                }
                if (LEVEL >= 2) doubt = doubt || (acc_s & ql.valid_rev) != ql.valid_rev;       // every data bin's decision must be trusted
                acc_i &= ql.valid_rev; acc_q &= ql.valid_rev;
                f_i += __popc(acc_i); f_q += __popc(acc_q); f_both += __popc(acc_i & acc_q);
            };
            if constexpr (NSYM2) { symbol(UnitIndex<2>{}, 0); symbol(UnitIndex<3>{}, 1); }
            else {
#pragma unroll 1
                for (int s = 0; s < n_sym; ++s) symbol(UnitIndex<0>{}, s);
            }
            float f_e2 = e2v.x + e2v.y;
            if (!active) { f_i = 0; f_q = 0; f_both = 0; f_e2 = 0.f; doubt = false; }
            // ---- frames whose decisions (checked) / tiny-|H| bins (EVM guard) are not provably the reference's: replayed whole
            uint32_t dm = __ballot_sync(0xffffffffu, doubt);
            while (dm != 0u) {                                    // warp-uniform: the whole warp replays one frame at a time
                const int g = (__ffs((int)dm) - 1) >> 3;
                dm &= ~(0xFFu << (8 * g));
                const long fr_id = f0 + g;
                const GlobalFrame<NSYM2 ? 2 : 0> fr = {p.in + fr_id * len, DRAWS ? p.g + fr_id * len : nullptr, p.tx_bits + fr_id * ((long)n_sym * 3), n_sym};
                const double sigma_d = NOISE != kNoiseNone ? __dsqrt_rn((double)__fdiv_rn(p.power[fr_id], p.snr_lin)) : 0.0;
                const ReplayTotals t = frame_replay_exact<NOISE>(fr, sigma_d, p.seed, p.stream, p.frame0 + (uint64_t)fr_id, ws.tile, &ws.lts[0][0], p.replayed);
                const uint32_t ti = __reduce_add_sync(0xffffffffu, t.i), tq = __reduce_add_sync(0xffffffffu, t.q);
                const uint32_t tb = __reduce_add_sync(0xffffffffu, t.both);
                float te2 = t.e2;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) te2 += __shfl_xor_sync(0xffffffffu, te2, o);
                if (grp == g) {                                   // lane 0 of the group books the frame
                    f_i = u == 0 ? ti : 0u; f_q = u == 0 ? tq : 0u; f_both = u == 0 ? tb : 0u;
                    f_e2 = u == 0 ? te2 : 0.f;
                }
            }
            f_e2 += __shfl_xor_sync(0xffffffffu, f_e2, 1);
            f_e2 += __shfl_xor_sync(0xffffffffu, f_e2, 2);
            f_e2 += __shfl_xor_sync(0xffffffffu, f_e2, 4);
            const uint32_t em = __ballot_sync(0xffffffffu, (f_i | f_q) != 0u);
            const bool mine = active && u == 0;
            const bool any_err = ((em >> (8 * grp)) & 0xFFu) != 0u;
            float evm;
            asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(evm) : "f"(f_e2 * inv_ref2));                                              // :1124
            a_i += f_i; a_q += f_q; a_both += f_both;
            a_ferr += (mine && any_err) ? 1u : 0u; a_frames += mine ? 1u : 0u;
            c_e2 += mine ? f_e2 : 0.f; c_evm += mine ? evm : 0.f;
        }
        a_e2 += (double)c_e2; a_evm += (double)c_evm;
    }
    if (p.counters == nullptr) return;
    const uint32_t t_i = warp_sum(a_i), t_q = warp_sum(a_q), t_both = warp_sum(a_both);
    const uint32_t t_ferr = warp_sum(a_ferr), t_frames = warp_sum(a_frames);
    const double t_e2 = warp_sum(a_e2), t_evm = warp_sum(a_evm);
    if (lane == 0) {
        s_cnt[warp][0] = (unsigned long long)t_i + 2ull * t_q - 2ull * t_both;     // bit errors (map of :423-430)
        s_cnt[warp][1] = (unsigned long long)t_i + t_q;
        s_cnt[warp][2] = t_ferr; s_cnt[warp][3] = t_frames;
        s_sum[warp][0] = t_e2; s_sum[warp][1] = t_evm;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long c[4] = {0, 0, 0, 0}; double sm[2] = {0, 0};
        for (int w = 0; w < WARPS; ++w) {
            for (int i = 0; i < 4; ++i) c[i] += s_cnt[w][i];
            for (int i = 0; i < 2; ++i) sm[i] += s_sum[w][i];
        }
        if (c[3] != 0) {
            ofdm_counters *o = p.counters;
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->bit_errors), c[0]);
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->rail_errors), c[1]);
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->frames_in_error), c[2]);
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->frames), c[3]);
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->bits), c[3] * 96ull * (unsigned long long)n_sym);
            atomicAdd(&o->sum_err2, sm[0]);
            atomicAdd(&o->sum_ref2, (double)c[3] * ref2_frame);
            atomicAdd(&o->sum_evm_lin, sm[1]);
        }
    }
}

}  // namespace ofdm
