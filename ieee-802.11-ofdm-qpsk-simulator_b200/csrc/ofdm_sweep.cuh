// ofdm_sweep.cuh -- the injected-noise SNR sweep of configs[1] (main()'s loop OFDM.c:1202-1222 over a batch of
// frames) in ONE kernel, k_sweep_lin.
//
// The sweep reuses each frame's draws g at every SNR point; only the scale sigma changes (OFDM.c:645-651).  The
// transform is linear, so   FFT(x + sigma g) = FFT(x) + sigma FFT(g):   a frame's four windows (LTS halves, two symbol
// bodies) and the matching four windows of draws are transformed ONCE, and every SNR point then costs one packed
// multiply-add per bin it needs -- F = X + sigma N for the lane's three data bins, G = (X_A + X_B) + sigma (N_A + N_B)
// for their channel estimates (:848; two per lane: two of its bins are the two symbols of one subcarrier) -- followed by
// the decision stage.  The frame and its draws cross HBM once per
// sweep instead of once per SNR point (3100 B per frame instead of 21 x 3100 B), the SNR loop touches neither shared
// memory nor the LSU, and the per-SNR totals live in registers of the lane that owns the SNR point (as in k_mc_philox).
//
// Exactness (OFDM_MODE_EXACT = kArithChecked) is the scheme of ofdm_chain.cuh: fp32 speculation, every rail decision
// verified against a rigorous bound on |speculated - reference|, doubtful (frame, SNR point)s replayed in the
// reference's arithmetic from global memory (stream_frame_replay).  The bound for this kernel, per bin of a window with
// clean samples x, draws g and S = |x|_2 + sigma |g|_2 (u = 2^-24; |X_k| <= 8 |x|_2 by Cauchy-Schwarz):
//   speculated  fl(X~ + sigma_f N~):  116 u |x|_2 + 116 u sigma |g|_2  (the two fp32 transforms, ofdm_chain.cuh)
//                                     + 8 u sigma |g|_2  (sigma_f = fl32(sigma_d))  + 8 u S  (rounding of the multiply-add)
//   reference   FFT_ref(x'), x' = fl(x + fl(sigma_d g)) (:651):  97 u |x'|_2 (its butterflies) + 8 (u sigma |g|_2 + u |x'|_2)
//                                     (the two roundings of x'), |x'|_2 <= S (1 + u)
//   channel estimate: + 32 u S for the reference's rounding of A + B, + 16 u S for fl(X~_A + X~_B), fl(N~_A + N~_B)
//   => within (116 + 8 + 8 + 97 + 16 + 32 + 16) u S = 293 u S <= kRadius S = 320 u S.
// A window's radius is therefore  kRadius |x|_2 + sigma kRadius |g|_2:  two norms per window per frame, one multiply-add
// per SNR point.  kArithFast keeps only the EVM guard (bins with a tiny channel estimate are replayed exactly).
#pragma once
#include "ofdm_chain.cuh"

namespace ofdm {

struct SweepParams {
    const float2 *in;               // TX frames [n_frames][320]
    const float *g;                 // injected standard normals [n_frames][320]
    const float *power;             // per-frame mean power (OFDM.c:637-643)
    const uint32_t *tx_bits;        // [n_frames][6]
    long n_frames;
    int n_snr;
    float radius_scale;             // kRadius, or infinity: every (frame, SNR point) is replayed exactly
    float evm_guard;                // EVM guard in radii (kEvmGuard; option "evm_guard")
    float snr_lin[kMaxSnr];         // (float)pow(10, snr/10), OFDM.c:645
    ofdm_counters *counters;        // [n_snr], accumulated into
    unsigned long long *replayed;   // the context's count of exactly replayed (frame, SNR point)s
};

struct alignas(16) SweepWarp {
    float2 tile[kWarpTile];         // transform transpose tile
    float2 fx[4][kWin];             // FFT of the clean windows: LTS half 1, LTS half 2, symbol 0, symbol 1 (natural bins)
    float2 fn[4][kWin];             // FFT of the draws of the same windows
    StreamStage<true> st[kStages];  // TMA ring: IQ windows + draw windows
    uint64_t bar[kStages];
    float norm[8];                  // kRadius |x_w|_2 (w = 0..3), kRadius |g_w|_2 (w = 0..3)
};
static_assert(sizeof(SweepWarp) % 16 == 0 && offsetof(SweepWarp, st) % 16 == 0 && offsetof(SweepWarp, norm) % 16 == 0, "SweepWarp alignment");

// |z| rounded up: approximate square root (2 ulps), rounding of the sum of squares, squares that underflow (below 1.1e-19
// in modulus: the floor term)
__device__ __forceinline__ float modulus_up(float2 z)
{
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(fmaf(z.x, z.x, z.y * z.y)));
    return fmaf(r, 1.000004f, 2e-19f);
}

// Which bins a lane takes (tools/deal_search.py sweep).  Symbols 0 and 1 of a subcarrier share the channel estimate
// G = A + B (:848), so each lane takes BOTH symbols of one "pair" bin -- items 0 and 1: one estimate, one |G|^2 and one
// reciprocal per SNR point for the two -- and one "single" item (item 2) of the 16 other bins: lanes 0..7 of a half-warp
// symbol 0, lanes 8..15 symbol 1 of the same 8 bins (as c_deal_bin).  The 16 pair bins of a half-warp are distinct mod 16, so
// their loads from all four tiles are conflict-free; the single items cost one extra wavefront per frame, the least
// possible (three of them fall on residue 2 mod 16 of the symbol tiles).
__constant__ unsigned char c_sweep_pair[32] = { 1,  2,  5,  8, 11, 16, 19, 41, 44, 45, 46, 52, 54, 55, 58, 63,
                                                3,  4, 10, 12, 17, 18, 22, 23, 25, 47, 48, 53, 56, 59, 61, 62};
__constant__ unsigned char c_sweep_single[16] = { 6, 14, 15, 20, 26, 40, 49, 50,    9, 13, 24, 38, 39, 42, 51, 60};

struct SweepItems {
    int bin[2];                     // natural FFT bin of estimate 0 (items 0 and 1) and of estimate 1 (item 2)
    int f_off[3];                   // where the item's bin sits in the symbol tiles fx[2..3]: sym*kWin + bin
    float k4[3];                    // 1 / sc = 4 * 0.5 L[bin]
    int word[3];                    // payload word of the frame holding the item's bit pair (sym*3 + d/16)
    int shift[3];                   // position of the pair in that word
};

__device__ __forceinline__ SweepItems make_sweep_items(int lane)
{
    SweepItems c;
    c.bin[0] = c_sweep_pair[lane];
    c.bin[1] = c_sweep_single[(lane >> 4) * 8 + (lane & 7)];
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const int bin = c.bin[t >> 1], sym = t == 2 ? (lane >> 3) & 1 : t;
        const int d = c_tab.bin_data[bin];
        c.f_off[t] = sym * kWin + bin;
        c.k4[t] = 4.f * (0.5f * (float)c_tab.bin_lts[bin]);
        c.word[t] = sym * 3 + (d >> 4);
        c.shift[t] = 2 * (d & 15);
    }
    return c;
}

// Block shape: 2 blocks of 6 warps per SM, in both arithmetics.  168 registers hold three SNR points per pass (nine
// independent item chains per warp) without spills, and 12 x 13.9 KB of shared memory fit.
constexpr int kSweepWarps = 6;

template <int ARITH>
__global__ void __launch_bounds__(kSweepWarps * 32, 2) k_sweep_lin(SweepParams p)
{
    constexpr int LEVEL = ARITH == kArithChecked ? 2 : 1;
    constexpr int kWarps = kSweepWarps;
    extern __shared__ __align__(128) unsigned char s_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, u = lane & 7;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);                  // same value, provably warp-uniform
    SweepWarp &ws = reinterpret_cast<SweepWarp *>(s_raw)[warp];
    SweepWarp &ws_u = reinterpret_cast<SweepWarp *>(s_raw)[warp_u];
    float2 *tile = ws.tile + grp * kGroupPitch;
    Tw<false> tw; tw.load(u);
    const SweepItems ic = make_sweep_items(lane);
    constexpr int len = 320;
    const long stride = (long)gridDim.x * kWarps;
    const long f_first = (long)blockIdx.x * kWarps + warp_u;
    const double q = (double)kQpsk;
    const double ref2_frame = 96.0 * (2.0 * q * q);
    const float inv_ref2 = (float)(1.0 / ref2_frame);
    constexpr uint32_t kBytes = 4 * 512 + 4 * 256;
    constexpr int kStep = 3;                          // SNR points per pass of the loop below

    const uint32_t stage0 = tma::saddr(&ws_u.st[0]);
    const uint32_t bar0 = tma::saddr(&ws_u.bar[0]);
    auto issue = [&](long f, int s) {          // f, s warp-uniform; whole warp calls (see k_stream_rx2)
        if (tma::elect_one()) {
            const uint32_t bar = bar0 + 8u * (uint32_t)s;
            const uint32_t dst = stage0 + (uint32_t)s * (uint32_t)sizeof(StreamStage<true>);
            const char *x = reinterpret_cast<const char *>(p.in) + f * (len * 8);
            const char *g = reinterpret_cast<const char *>(p.g) + f * (len * 4);
            const uint32_t gd = dst + 4 * kWin * 8;
            tma::expect_tx_addr(bar, kBytes);
            tma::bulk_addr(dst + 0 * kWin * 8, x + 32 * 8, 512, bar);             // Channel_Estimation :837
            tma::bulk_addr(dst + 1 * kWin * 8, x + 96 * 8, 512, bar);             //                    :838
            tma::bulk_addr(dst + 2 * kWin * 8, x + 176 * 8, 512, bar);            // CP strip :1028, symbol 0
            tma::bulk_addr(dst + 3 * kWin * 8, x + 256 * 8, 512, bar);            //                 symbol 1
            tma::bulk_addr(gd + 0 * kWin * 4, g + 32 * 4, 256, bar);
            tma::bulk_addr(gd + 1 * kWin * 4, g + 96 * 4, 256, bar);
            tma::bulk_addr(gd + 2 * kWin * 4, g + 176 * 4, 256, bar);
            tma::bulk_addr(gd + 3 * kWin * 4, g + 256 * 4, 256, bar);
        }
    };
    if (lane == 0) {
        for (int s = 0; s < kStages; ++s) tma::mbar_init(&ws.bar[s], 1);
        tma::fence_mbar_init();
    }
    __syncwarp();
    for (int s = 0; s < kStages; ++s)
        if (f_first + s * stride < p.n_frames) issue(f_first + s * stride, s);

    // Per-SNR totals live in registers: lane L owns SNR points L and L + 32 (n_snr <= 64).  The float EVM sums are
    // flushed into doubles every 64 frames.
    uint32_t m_i[2] = {0, 0}, m_q[2] = {0, 0}, m_b[2] = {0, 0}, m_ferr[2] = {0, 0};
    float m_e2[2] = {0.f, 0.f}, m_evm[2] = {0.f, 0.f};
    double d_e2[2] = {0.0, 0.0}, d_evm[2] = {0.0, 0.0};
    uint32_t n_done = 0;
    uint32_t k = 0;                                   // frames this warp has consumed (ring position)
    for (long f = f_first; f < p.n_frames; f += stride, ++k) {
        const int s = (int)(k & 1u);
        const uint32_t phase = (k >> 1) & 1u;
        // global loads first; what depends on them (noise scales, bit pairs) is computed after the transforms, which hide their latency
        const float P = p.power[f];
        const uint32_t *wb = p.tx_bits + f * 6;
        uint32_t txw[3];
#pragma unroll
        for (int t = 0; t < 3; ++t) txw[t] = wb[ic.word[t]];

        tma::wait_addr(bar0 + 8u * (uint32_t)s, phase);
        float2 v[8];
        float gz[8];
        float2 n2x = make_float2(0.f, 0.f);
        float n2g = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            v[i] = ws.st[s].x[grp][u + 8 * i];
            gz[i] = ws.st[s].g[grp][u + 8 * i];
            n2x = __ffma2_rn(v[i], v[i], n2x);
            n2g = fmaf(gz[i], gz[i], n2g);
        }
        __syncwarp();                                         // every lane has its samples: the stage can be refilled
        if (f + kStages * stride < p.n_frames) issue(f + kStages * stride, s);
        fft64<false>(v, tw, tile, u);                         // X = FFT(x window)
#pragma unroll
        for (int j = 0; j < 8; ++j) ws.fx[grp][u + 8 * j] = v[j];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = make_float2(gz[i], 0.f);     // the noise is real-rail only (SURVEY Q1)
        fft64<false>(v, tw, tile, u);                         // N = FFT(g window)
#pragma unroll
        for (int j = 0; j < 8; ++j) ws.fn[grp][u + 8 * j] = v[j];
        // window norms |x_w|_2, |g_w|_2 over the group's 8 lanes -> error radii per unit of (1, sigma)
        float2 nn = make_float2(n2x.x + n2x.y, n2g);
#pragma unroll
        for (int o = 1; o < 8; o <<= 1)
            nn = __fadd2_rn(nn, make_float2(__shfl_xor_sync(0xffffffffu, nn.x, o), __shfl_xor_sync(0xffffffffu, nn.y, o)));
        {
            float rx, rn;
            asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rx) : "f"(nn.x));
            asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rn) : "f"(nn.y));
            const bool ok = nn.x >= 1e-30f && nn.x < 1e20f && nn.y < 1e20f;      // NaN fails; all-zero draws are fine
            const float inf = __int_as_float(0x7f800000);
            if (u == 0) { ws.norm[grp] = ok ? p.radius_scale * rx : inf; ws.norm[4 + grp] = ok ? p.radius_scale * rn : inf; }
        }
        __syncwarp();
        // the lane's three data bins and their two channel estimates: everything the SNR loop needs, in registers
        const float4 rX = *reinterpret_cast<const float4 *>(ws.norm), rN = *reinterpret_cast<const float4 *>(ws.norm + 4);
        const float rHX = rX.x + rX.y, rHN = rN.x + rN.y;                      // 2 r_H = r_A + r_B
        float2 FX[3], FN[3], GX[2], GN[2];
        float c0[3], c1[3], c2[3], hcX[2], hcN[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int bin = ic.bin[e];
            GX[e] = cadd(ws.fx[0][bin], ws.fx[1][bin]);                        // A + B (:848), clean part
            GN[e] = cadd(ws.fn[0][bin], ws.fn[1][bin]);                        //               noise part
            if (LEVEL >= 2) { hcX[e] = modulus_up(GX[e]); hcN[e] = modulus_up(GN[e]); }
        }
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            FX[t] = (&ws.fx[2][0])[ic.f_off[t]];
            FN[t] = (&ws.fn[2][0])[ic.f_off[t]];
            const bool sym0 = ic.f_off[t] < kWin;                              // the item's symbol
            const float rFX = sym0 ? rX.z : rX.w, rFN = sym0 ? rN.z : rN.w;
            // The decision threshold, r_F (|G| + r_H2) + r_H2 |F| + 2u |F| |G| (the numerator F conj(G) moves by at most
            // |dF||G| + |F||dG| + |dF||dG| in either rail, and its fp32 evaluation errs by at most 2u (|ac| + |bd|) <= 2u |F||G|:
            // Cauchy-Schwarz, moduli instead of the 1-norms process_bin_spec uses per point), as a polynomial in sigma: with
            // |F| <= |FX| + sigma |FN|, |G| <= |GX| + sigma |GN| (triangle inequality) and the radii r = rX + sigma rN, every
            // factor is a non-negative affine function of sigma, so the products are bounded by c0 + c1 sigma + c2 sigma^2 --
            // three coefficients per item and frame, two multiply-adds per SNR point.  The moduli are rounded up (approximate
            // square root, squares that underflow: windows below 1e-15 in norm are never speculated, so 2e-19 covers them).
            if (LEVEL >= 2) {
                const float faX = modulus_up(FX[t]), faN = modulus_up(FN[t]);
                const float hX = hcX[t >> 1], hN = hcN[t >> 1];
                const float A0 = hX + rHX, A1 = hN + rHN;
                c0[t] = fmaf(rFX, A0, fmaf(rHX, faX, 1.2e-7f * (faX * hX)));
                c1[t] = fmaf(rFX, A1, fmaf(rFN, A0, fmaf(rHX, faN, fmaf(rHN, faX, 1.2e-7f * fmaf(faX, hN, faN * hX)))));
                c2[t] = fmaf(rFN, A1, fmaf(rHN, faN, 1.2e-7f * (faN * hN)));
            } else { c0[t] = c1[t] = c2[t] = 0.f; }
        }
        __syncwarp();                                         // everyone holds its items: fx / fn may be overwritten
        // Fold the transmitted rails' signs and the sign of sc into the items (exact: negations commute with every rounding).
        // With S = F conj(G): negating F.x and G.y negates S.x alone, negating F.y and G.y negates S.y alone, so after
        //   F.x ^= (tx I-rail sign ^ sign sc),  F.y ^= (tx Q-rail sign ^ sign sc),  G.y ^= (tx I-rail sign ^ tx Q-rail sign)
        // every item looks as if (+1, +1)/sqrt(2) had been sent through sc = +1/2: a rail error is the sign bit of S, the error
        // vector is 2 S / |G|^2 - (h, h), and |G|^2, the moduli and the thresholds are unchanged.  Item 1 shares item 0's
        // estimate: its G.y differs from item 0's by the sign g_rel, applied per point.  The replay reads global memory.
        uint32_t gq[3];
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            const uint32_t tp = txw[t] >> ic.shift[t];
            const uint32_t kb = __float_as_uint(ic.k4[t]) & 0x80000000u;
            const uint32_t fq = (tp << 31) ^ kb, fi = ((tp ^ (tp >> 1)) << 31) ^ kb;
            gq[t] = (tp >> 1) << 31;
            FX[t] = make_float2(__uint_as_float(__float_as_uint(FX[t].x) ^ fi), __uint_as_float(__float_as_uint(FX[t].y) ^ fq));
            FN[t] = make_float2(__uint_as_float(__float_as_uint(FN[t].x) ^ fi), __uint_as_float(__float_as_uint(FN[t].y) ^ fq));
        }
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            GX[e].y = __uint_as_float(__float_as_uint(GX[e].y) ^ gq[2 * e]);
            GN[e].y = __uint_as_float(__float_as_uint(GN[e].y) ^ gq[2 * e]);
        }
        const uint32_t g_rel = gq[0] ^ gq[1];
        // the noise scale of every SNR point, (float)sqrt((double)(P / snr)) (:647, :651), one (two) per lane
        // (the double square root rounded to float is the correctly rounded float square root: 53 >= 2 * 24 + 2 bits, so the
        // second rounding cannot change the result -- no double arithmetic needed here; the replay takes sigma in double)
        float sig_lo = 0.f, sig_hi = 0.f;
        if (lane < p.n_snr) sig_lo = __fsqrt_rn(__fdiv_rn(P, p.snr_lin[lane]));
        if (p.n_snr > 32 && lane + 32 < p.n_snr) sig_hi = __fsqrt_rn(__fdiv_rn(P, p.snr_lin[lane + 32]));
        // ... through shared memory (a free noise tile): one broadcast load per pass in the loop.  Three points per pass sit
        // in one 16-byte slot (points 3i..3i+2 at 4i..4i+2); the slots past n_snr hold 0.
        auto sig_pos = [](int i) { return (i / 3) * 4 + i % 3; };
        float *sigs = reinterpret_cast<float *>(&ws.fn[1][0]);
        sigs[sig_pos(lane)] = sig_lo; sigs[sig_pos(lane + 32)] = sig_hi;
        if (lane < 2) sigs[sig_pos(64 + lane)] = 0.f;
        __syncwarp();

        // ---- SNR loop OFDM.c:1202: one packed multiply-add per value, then the decision stage.  Per-point results
        // {packed rail errors, sum |e|^2} go through 64 words of shared memory (the noise tiles are free by now and the
        // replay does not touch them) so that the owner lanes book them once per frame instead of branching per point.
        // The loop body has no data-dependent branch: each lane collects its doubtful points in a bit mask, and the warp
        // resolves them after the loop (one vote per frame), patching their words before they are booked.
        uint2 *res = reinterpret_cast<uint2 *>(&ws.fn[0][0]);
        const float g2_limit = p.radius_scale * 1.58e6f;        // 8 rH2 / radius_scale (1 + 1e-4) < sqrt(1.6e14); infinite radius: never
        // one SNR point is prepared (noise scale, channel radius, guards) and then evaluated item by item, so that the loop body
        // below can place the steps of the previous pass's warp reduction between the items
        struct PointState { float sg, rH2, den_min4; float2 e2v; uint32_t pk; bool doubt; float2 G; float den, inv; };
        auto point_begin = [&](float sg) {
            PointState q;
            q.sg = sg;
            q.rH2 = fmaf(sg, rHN, rHX);
            const float gd = p.evm_guard * q.rH2;
            q.den_min4 = gd * gd;
            q.e2v = make_float2(0.f, 0.f);
            // every bin of G = A + B is at most 8 (|x_A| + sigma |g_A| + |x_B| + sigma |g_B|) = 8 rH2 / radius_scale in modulus:
            // |G|^2 < 1.6e14 (the reference's quotient cannot overflow, process_bin_spec) is checked once per point
            q.pk = 0; q.doubt = !(q.rH2 < g2_limit);
            return q;
        };
        auto point_item = [&](PointState &q, int t) {                                    // straight-line: no votes, no branches
            const float2 sg2 = make_float2(q.sg, q.sg);
            if (t != 1) {                                     // items 0 and 2 form their estimate, item 1 uses item 0's
                q.G = __ffma2_rn(sg2, GN[t >> 1], GX[t >> 1]);
                q.den = fmaf(q.G.x, q.G.x, q.G.y * q.G.y);
                asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(q.inv) : "f"(q.den));
            }
            const float2 G = t == 1 ? make_float2(q.G.x, __uint_as_float(__float_as_uint(q.G.y) ^ g_rel)) : q.G;
            const float2 F = __ffma2_rn(sg2, FN[t], FX[t]);
            const float thr = fmaf(fmaf(c2[t], q.sg, c1[t]), q.sg, c0[t]);
            q.pk += process_bin_spec_den<LEVEL, true>(F, G, q.den, q.inv, 2.f, 0u, thr, q.rH2, q.den_min4, q.e2v, q.doubt);
        };
        // The warp sums of a pass (one REDUX per point for the packed counts, five dependent shuffle steps for the sums |e|^2)
        // are finished one iteration late, on top of the next pass's nine independent item chains.
        uint32_t pk_raw[kStep];                                 // the previous pass's per-lane packed counts and sums |e|^2
        float e2_pend[kStep], red[kStep], red_in[kStep];
#pragma unroll
        for (int j = 0; j < kStep; ++j) { pk_raw[j] = 0; e2_pend[j] = 0.f; }
        auto red_issue = [&](int o) {
#pragma unroll
            for (int j = 0; j < kStep; ++j) red_in[j] = __shfl_xor_sync(0xffffffffu, red[j], o);
        };
        auto red_take = [&]() {
#pragma unroll
            for (int j = 0; j < kStep; ++j) red[j] += red_in[j];
        };
        uint64_t doubt_mask = 0;                                // the lane's doubtful points
        for (int si = 0, sk = 0; si < p.n_snr; si += kStep, sk += 4) {
            uint32_t pk_sum[kStep];
#pragma unroll
            for (int j = 0; j < kStep; ++j) { pk_sum[j] = __reduce_add_sync(0xffffffffu, pk_raw[j]); red[j] = e2_pend[j]; }   // the three 8-bit fields stay below 97
            red_issue(16);
            PointState q[kStep];
            const float4 sp = *reinterpret_cast<const float4 *>(sigs + sk);
            q[0] = point_begin(sp.x); q[1] = point_begin(sp.y); q[2] = point_begin(sp.z);
            // item n of the pass, then the next shuffle step: offsets 8, 4, 2, 1 after the first four items
#pragma unroll
            for (int t = 0; t < 3; ++t) {
#pragma unroll
                for (int j = 0; j < kStep; ++j) {
                    const int n = t * kStep + j;
                    point_item(q[j], t);
                    if (n < 4) { red_take(); red_issue(8 >> n); }
                    else if (n == 4) red_take();
                }
            }
            if (lane == 0 && si > 0) {
#pragma unroll
                for (int j = 0; j < kStep; ++j) res[si - kStep + j] = make_uint2(pk_sum[j], __float_as_uint(red[j]));
            }
            uint32_t bits = 0;
#pragma unroll
            for (int j = 0; j < kStep; ++j) {
                pk_raw[j] = q[j].pk;
                e2_pend[j] = q[j].e2v.x + q[j].e2v.y;
                bits |= (uint32_t)q[j].doubt << j;
            }
            doubt_mask |= (uint64_t)bits << si;
        }
        {
            const int last = (p.n_snr - 1) / kStep * kStep;                              // first point of the last pass
#pragma unroll
            for (int j = 0; j < kStep; ++j) {
                const uint32_t pk_sum = __reduce_add_sync(0xffffffffu, pk_raw[j]);
                float r = e2_pend[j];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
                if (lane == 0) res[last + j] = make_uint2(pk_sum, __float_as_uint(r));   // up to res[65]: inside the tile
            }
        }
        // ---- the doubtful points (rare): whole warp, one point at a time
        {
            if (p.n_snr < 64) doubt_mask &= (1ull << p.n_snr) - 1ull;                    // the points past the end of the last pass
            uint64_t todo = __reduce_or_sync(0xffffffffu, (uint32_t)doubt_mask);
            if (p.n_snr > 32) todo |= (uint64_t)__reduce_or_sync(0xffffffffu, (uint32_t)(doubt_mask >> 32)) << 32;
            __syncwarp();                                                                // lane 0's words are written
            while (todo != 0) {                                                          // warp-uniform
                const int si = __ffsll((long long)todo) - 1;
                todo &= todo - 1;
                const float sg = sigs[sig_pos(si)];
                bool replay = true;
                if (LEVEL >= 2) {
                    // The polynomial is an upper bound of the per-point threshold (triangle inequality): before paying for a
                    // replay, recheck the point with the threshold of its actual |F|, |G|.
                    const float4 qX = *reinterpret_cast<const float4 *>(ws.norm), qN = *reinterpret_cast<const float4 *>(ws.norm + 4);
                    const float2 sg2 = make_float2(sg, sg);
                    const float rH2 = fmaf(sg, rHN, rHX);
                    const float gd = p.evm_guard * rH2, den_min4 = gd * gd;
                    bool doubt2 = false;
                    float2 e2w = make_float2(0.f, 0.f);
                    float2 G;
#pragma unroll
                    for (int t = 0; t < 3; ++t) {
                        if (t != 1) G = __ffma2_rn(sg2, GN[t >> 1], GX[t >> 1]);
                        const float2 Gt = t == 1 ? make_float2(G.x, __uint_as_float(__float_as_uint(G.y) ^ g_rel)) : G;
                        const float2 F = __ffma2_rn(sg2, FN[t], FX[t]);
                        const bool sym0 = ic.f_off[t] < kWin;
                        const float rF = fmaf(sg, sym0 ? qN.z : qN.w, sym0 ? qX.z : qX.w);
                        const float fa = modulus_up(F), hc = modulus_up(Gt);
                        const float thr = fmaf(rF, hc + rH2, fmaf(rH2, fa, 1.2e-7f * (fa * hc)));
                        process_bin_spec<LEVEL, true>(F, Gt, 2.f, 0u, thr, rH2, den_min4, e2w, doubt2);
                    }
                    replay = __any_sync(0xffffffffu, doubt2);
                }
                if (replay) {                                 // not provably the reference's decisions / EVM: replay exactly
                    const double sigma_d = __dsqrt_rn((double)__fdiv_rn(P, p.snr_lin[si]));
                    const uint2 r = stream_frame_replay<kNoiseInject>(p.in + f * len, p.g + f * len, wb, sigma_d, 0u, 0u, 0ull,
                                                                      ws.tile, &ws.fx[0][0], p.replayed);
                    const uint32_t pk_sum = __reduce_add_sync(0xffffffffu, r.x);
                    float e2 = __uint_as_float(r.y);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) e2 += __shfl_xor_sync(0xffffffffu, e2, o);
                    if (lane == 0) res[si] = make_uint2(pk_sum, __float_as_uint(e2));
                }
            }
        }
        __syncwarp();
        // the lane that owns an SNR point books the frame's result for it (lanes beyond n_snr read stale words and add nothing)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (h == 1 && p.n_snr <= 32) break;                                         // warp-uniform: no second half to book
            const uint2 r = res[lane + 32 * h];
            const bool mine = lane + 32 * h < p.n_snr;
            const uint32_t pk = mine ? r.x : 0u;
            const float e2 = mine ? __uint_as_float(r.y) : 0.f;
            float evm;
            asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(evm) : "f"(e2 * inv_ref2));                 // :1124
            m_i[h] += pk & 0xFFu; m_q[h] += (pk >> 8) & 0xFFu; m_b[h] += pk >> 16; m_ferr[h] += pk != 0u;
            m_e2[h] += e2; m_evm[h] += evm;
        }
        n_done += 1;
        if ((n_done & 63u) == 0u) {
#pragma unroll
            for (int h = 0; h < 2; ++h) { d_e2[h] += (double)m_e2[h]; d_evm[h] += (double)m_evm[h]; m_e2[h] = 0.f; m_evm[h] = 0.f; }
        }
    }
    if (n_done == 0) return;
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

inline size_t sweep_smem_bytes(int warps) { return sizeof(SweepWarp) * warps; }

}  // namespace ofdm
