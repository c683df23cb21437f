// ofdm_chain.cuh -- fused whole-chain kernels for the default frame shape (LTS + 2 data symbols,
// OFDM.c:20,439: the reference message gives data_frames_number = 2).
//
// A warp owns one frame at a time: its four 8-lane groups transform LTS half 1, LTS half 2, data
// symbol 0 and data symbol 1 in one pass (see ofdm_device.cuh).  After the transform the 96 data
// bins of the two symbols are dealt out evenly, three per lane, for equalise / slice / demod / EVM /
// BER ("items"), so no lane idles on null or pilot bins and nothing is selected per bin at run time:
// every per-item constant (which bin, which L sign, which payload word and bit) is fixed per lane.
//
//   k_mc_philox   Monte-Carlo sweep with nothing in HBM but the counters: payload bits and the noise
//                 come from Philox4x32-10 streams, the frame is built in shared memory once and reused
//                 for every SNR point of the sweep.
#pragma once
#include "ofdm_kernels.cuh"

namespace ofdm {

constexpr int kWin = 72;            // skewed pitch of a 64-sample window in shared memory (bank-conflict-free groups)
constexpr int kMaxSnr = 64;
constexpr int kMaxTaps = 16;

struct ItemConst {
    int f_off[3];                   // where the item's FFT output sits in the F exchange tile: sym*kWin + bin
    int bin[3];                     // natural FFT bin (index into the LTS exchange tiles)
    float sc[3];                    // 0.5 * L[bin]
    int word[3];                    // payload word of the frame holding the item's bit pair (sym*3 + d/16)
    int shift[3];                   // position of the pair in that word
};

// Which of the frame's 96 data bins a lane takes.  The exchange tiles are read with 64-bit loads, one half-warp (16 lanes) per
// shared-memory wavefront: a load is conflict-free when the 16 lanes touch 16 different bank pairs (element index mod 16) or
// the same address.  Dealing the data indices out in order (item t = lane + 32 r) cannot achieve that -- 16 consecutive data
// bins span 17 or 18 FFT bins because of the pilot / DC gaps, so two of them always collide (18 extra wavefronts per frame).
// Instead each half-warp takes 8 bins for BOTH symbols (lanes 0..7 symbol 0, lanes 8..15 symbol 1): the LTS tiles are then
// read at 8 addresses, each by two lanes (a broadcast), and the symbol tiles sit 72 = 8 (mod 16) elements apart, so the bins
// of a group only have to differ mod 8 -- which the table below (found by search, tools/deal_search.py) achieves for all
// groups but one: 1 extra wavefront per frame instead of 18.  Row = 2 r + half-warp.
__constant__ unsigned char c_deal_bin[48] = { 2, 10, 12, 14, 16, 23, 49, 54,    1,  3, 18, 40, 46, 60, 61, 63,   22, 25, 45, 47, 48, 50, 52, 59,
                                              4,  6,  9, 11, 13, 24, 39, 58,    8, 41, 42, 44, 51, 53, 55, 62,    5, 15, 17, 19, 20, 26, 38, 56};

__device__ __forceinline__ ItemConst make_items(int lane)
{
    ItemConst c;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int sym = (lane >> 3) & 1;
        const int bin = c_deal_bin[(2 * r + (lane >> 4)) * 8 + (lane & 7)];
        const int d = c_tab.bin_data[bin];
        c.f_off[r] = sym * kWin + bin;
        c.bin[r] = bin;
        c.sc[r] = 0.5f * (float)c_tab.bin_lts[bin];
        c.word[r] = sym * 3 + (d >> 4);
        c.shift[r] = 2 * (d & 15);
    }
    return c;
}

// One data bin (see process_bin_hot in ofdm_kernels.cuh for the exactness argument): returns the
// rail errors packed as  I | Q << 8 | both << 16  and adds |E - tx|^2 to e2.
template <bool EXACT>
__device__ __forceinline__ uint32_t item_eval(float2 F, float2 Hh, float sc, uint32_t txp, float &e2)
{
    return process_bin_hot<EXACT>(F, Hh, sc, txp, true, e2);
}

// ---- arithmetic of the fused kernels (streaming receiver, Monte-Carlo) ----------------------------
//   kArithFast     fp32 transform, fp32 channel, fp32 decisions
//   kArithExact    the reference's arithmetic everywhere (ofdm_device.cuh, EXACT mode)
//   kArithChecked  what OFDM_MODE_EXACT runs for the sweep: channel in the reference's arithmetic (so the
//                  noisy time samples are the reference's bit for bit), transform and decisions speculated in
//                  fp32, every decision verified against a rigorous bound on |fp32 path - reference path|,
//                  and the whole frame replayed in the reference's arithmetic when any of its 192 rail
//                  decisions is not provably the reference's.  Error counts are therefore exactly those of
//                  kArithExact; the EVM sums differ by fp32 rounding (1e-5 contract), as they already do there.
//
// The bound.  Both transforms compute the same DFT of the same 64 floats x (u = 2^-24).  A radix-2 stage is sqrt(2) times a
// unitary map: an error introduced after stage s, of norm e |v_s|_2 with |v_s|_2 = 2^(s/2) |x|_2, reaches the output with
// norm 2^((6-s)/2) e |v_s|_2 = 8 e |x|_2, whatever the stage, and no bin errs by more than the norm of the error vector.
//   Reference (OFDM.c:282-312): per stage the double product w*b rounded to float (<= u(1 + 2^-26) |b|), then a float
//   add (<= u |v_out|): 6 * 2u * 8 |x|_2 <= 97 u |x|_2.
//   fp32 path (fft64_fast = dft8, twiddles, transpose, dft8; ofdm_device.cuh), stage by stage:
//     dft8: three stages of complex additions (u |v_out| each; the factors -i are swaps and sign changes, exact) and one
//           diagonal step on two of the eight values, b * W8^(1,3) = fl(fl(x +- y) * fl(sqrt(1/2))): (1+u)^2 (1 + 0.29u),
//           <= 2.3 u |b|                                                                        ->  5.3 u   (5.5 charged)
//     twiddles: cmul = (fma(a.x, b.x, -fl(a.y b.y)), fma(a.x, b.y, fl(a.y b.x))): componentwise u(|a.x b.x| + 2|a.y b.y|),
//           u(|a.x b.y| + 2|a.y b.x|), so <= sqrt(5) u |a||b| in modulus; the float twiddle is within u of the true one
//                                                                                               ->  3.3 u
//     total (5.5 + 3.3 + 5.5) * 8 u |x|_2 = 114.4, charged as 116 u |x|_2.
//   (Round 1 charged every fp32 stage 5u: 272 u.  The per-stage count above is what the code does.)
// The channel estimate adds the rounding of A + B (:848): <= 2u |A + B| <= 32 u max(|x_A|_2, |x_B|_2).  Every bin of a
// window is therefore within
//      radius = kRadius * |x|_2,   kRadius = 320 u  (>= 97 + 116 + 32 (+ 32, below) = 277, the rest is margin for the
// second-order terms, the approximate square root and the rounding of the threshold itself)
// of the reference's value, for F, and (radius_A + radius_B)/2 for H.  With F = F~ + dF, H = H~ + dH the numerator
// of the equaliser (:1050) moves by at most |dF| |H|_1 + |dH| |F|_1 + |dF||dH|, and its fp32 evaluation errs by
// 2^-23 |F|_1 |H|_1 more (process_bin_hot).  The decision (:860-868) is the sign of the reference's numerator
// whenever the quotient cannot underflow, which the magnitude guards below ensure.
//
// The channel is speculated too (round 2): the kernel adds the noise as fma(sigma_f, g, x) with sigma_f = (float)sigma_d,
// the reference as fl32(x + fl32(sigma_d * g)) (:651).  Per sample the two differ by at most 2u |sigma g| + 2u |x'|
// (rounding of sigma, of the product, of the two sums), so for a window |delta|_2 <= 2u |sigma g|_2 + 2u |x'|_2
// <= 4u |x'|_2 + 2u |x|_2 with x the clean samples, and the transform maps it to at most 8 |delta|_2 in any bin:
// 32 u |x'|_2, charged to kRadius (97 + 116 + 32 + 32 = 277 <= 320), plus 16 u |x|_2 <= 16 u sqrt(len * P), P the
// frame's mean power of :637-643 -- the kChanRadius term (18 u, margin included), which does not depend on the window.
enum { kArithFast = 0, kArithExact = 1, kArithChecked = 2 };
constexpr float kRadius = 320.f * 5.9604645e-8f;
constexpr float kChanRadius = 18.f * 5.9604645e-8f;

// frames the speculating kernels replayed exactly are counted per context (a device word owned by the ofdm_ctx, passed in the
// kernel parameters as `replayed`)

// radius of one window from the lane's share of sum |x|^2; windows whose energy is outside [1e-30, 1e20] are never
// trusted (squares may have underflowed / the magnitude guards of the decision would not hold)
__device__ __forceinline__ float window_radius(float2 n2v, float scale, float extra)
{
    float n2 = n2v.x + n2v.y;
    n2 += __shfl_xor_sync(0xffffffffu, n2, 1);
    n2 += __shfl_xor_sync(0xffffffffu, n2, 2);
    n2 += __shfl_xor_sync(0xffffffffu, n2, 4);
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(n2));          // flushing is harmless: n2 < 1e-30 is rejected
    return (n2 >= 1e-30f && n2 < 1e20f) ? fmaf(scale, r, extra) : __int_as_float(0x7f800000);
}

// One data bin, speculated: like process_bin_hot<false>, and reports whether both rail decisions are provably the
// reference's.  rF / rH: error radii of F and H.  den_min: bins whose |H|^2 is below it are not trusted either --
// not for the decisions but for the EVM sum, which at low SNR is dominated by the few bins with a tiny estimate
// (|E|^2 ~ 1/|H|^2), where the fp32 transform's error in H would show: with |H| >= kEvmGuard radii the relative
// error of an accepted quotient stays below ~1e-5 for the rarest accepted bins (the bound is about 200x the typical
// error) and the sums agree with the all-exact kernel's to ~1e-7 (4x the guard: 1e-8, at 4x the replays on fading channels).
// 820 radii of 320 u = the 512 radii of 512 u of the first round-2 builds: the guard is about typical errors, not the bound.
constexpr float kEvmGuard = 820.f;
//
// The estimate comes in unscaled, G = A + B with H = sc G, sc = +-0.5 (:848): powers of two commute with every rounding
// here, so the test is done on G (numerator, thresholds and guards scaled accordingly, rH2 = 2 rH) and the quotient
// is recovered with k = 4 sc = 1 / sc ... E = F conj(G) / |G|^2 * k; the sign of sc joins the sign comparison.
// LEVEL 2: decisions and EVM guard verified (kArithChecked).  LEVEL 1: EVM guard only -- what the fast kernels of round 2 use
// so that their EVM sums stay within 1e-5 of the reference's too (the rare frames with a tiny |H| bin are replayed exactly).
// THR_GIVEN: the caller supplies the decision threshold (rF carries it; rH2 unused) -- the sweep kernel evaluates it as a
// polynomial in sigma per item instead of from |F|_1 and |G|_1 per point (ofdm_sweep.cuh) -- and has bounded |G|^2 < 1.6e14
// for the whole frame from the window norms.
// process_bin_spec_den takes |G|^2 = fma(G.x, G.x, G.y * G.y) and its approximate reciprocal from the caller, which may share
// them between bins with the same estimate (the sweep kernel: both symbols of a subcarrier).
template <int LEVEL, bool THR_GIVEN = false>
__device__ __forceinline__ uint32_t process_bin_spec_den(float2 F, float2 G, float den, float inv, float k, uint32_t txp, float rF,
                                                         float rH2, float den_min4, float2 &e2, bool &doubt)
{
    const float a = F.x, b = F.y, c = G.x, d = G.y;
    // numerator F * conj(G) = (fma(a, c, b*d), fma(b, c, -(a*d))) in two packed instructions
    const float2 pt = __fmul2_rn(make_float2(d, d), make_float2(b, a));
    const float2 S = __ffma2_rn(make_float2(c, c), F, make_float2(pt.x, -pt.y));
    const float sr = S.x, si = S.y;
    const uint32_t sq = txp << 31, sx = (txp ^ (txp >> 1)) << 31;          // IEEE sign bits of the tx Q / I rails
    const uint32_t kb = __float_as_uint(k);
    const uint32_t ei_ = (__float_as_uint(sr) ^ sx ^ kb) >> 31, eq_ = (__float_as_uint(si) ^ sq ^ kb) >> 31;
    bool safe;
    if (LEVEL >= 2) {
        float thr;
        if (THR_GIVEN) thr = rF;
        else {
            const float fa = fabsf(a) + fabsf(b), hc = fabsf(c) + fabsf(d);
            thr = fmaf(rF, hc + rH2, fmaf(rH2, fa, 1.2e-7f * (fa * hc)));
        }
        // reference numerator >= 1e-30 in magnitude and reference |H|^2 < 1e14: the float quotient keeps its sign (>= 1e-44)
        // THR_GIVEN callers have checked den < 1.6e14 for all bins of the frame at once (from the window norms)
        safe = (fminf(fabsf(sr), fabsf(si)) - thr) > 2e-30f && (THR_GIVEN || den < 1.6e14f) && den > den_min4;
    } else {
        safe = (THR_GIVEN || den < 1.6e14f) && den > den_min4;
    }
    doubt = doubt || !safe;
    // E - tx = (S * inv) * k - (+-1/sqrt(2)); e2 collects the squares of the two rails separately (summed per frame)
    const float2 U = __fmul2_rn(S, make_float2(inv, inv));
    const float2 D = __ffma2_rn(U, make_float2(k, k), make_float2(__uint_as_float(0xBF3504F3u ^ sx), __uint_as_float(0xBF3504F3u ^ sq)));
    e2 = __ffma2_rn(D, D, e2);
    return ei_ | (eq_ << 8) | ((ei_ & eq_) << 16);
}
template <int LEVEL, bool THR_GIVEN = false>
__device__ __forceinline__ uint32_t process_bin_spec(float2 F, float2 G, float k, uint32_t txp, float rF, float rH2, float den_min4,
                                                     float2 &e2, bool &doubt)
{
    const float den = fmaf(G.x, G.x, G.y * G.y);
    float inv;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(den));
    return process_bin_spec_den<LEVEL, THR_GIVEN>(F, G, den, inv, k, txp, rF, rH2, den_min4, e2, doubt);
}
__device__ __forceinline__ uint32_t process_bin_checked(float2 F, float2 G, float k, uint32_t txp, float rF, float rH2, float den_min4,
                                                        float2 &e2, bool &doubt)
{
    return process_bin_spec<2>(F, G, k, txp, rF, rH2, den_min4, e2, doubt);
}

struct McParams {
    uint32_t seed;
    uint64_t frame0;
    long n_frames;
    int n_snr;
    float snr_lin[kMaxSnr];         // (float)pow(10, snr/10), OFDM.c:645
    float inv_sqrt_snr[kMaxSnr];    // 1/sqrt(snr_lin), fast mode's noise scale factor
    uint32_t stream[kMaxSnr];       // Philox noise stream of each point (the index of the SNR point in the caller's full list)
    float radius_scale;             // kArithChecked: kRadius, or infinity to replay every point
    float radius_chan;              // kArithChecked: kChanRadius * sqrt(320) (times sqrt(P) = the channel term), or infinity
    float evm_guard;                // EVM guard in radii (kEvmGuard; option "evm_guard")
    int n_taps;                     // multipath variant: taps per frame (1..kMaxTaps)
    ofdm_counters *counters;        // [n_snr], accumulated into
    unsigned long long *replayed;   // the context's count of exactly replayed (frame, SNR point)s
};

// per-warp shared memory of the fused kernels
struct WarpShared {
    float2 tile[kWarpTile];         // transform transpose tile, then the F exchange tile (2 x kWin used)
    float2 lts[2][kWin];            // FFT of the two received LTS halves
    float2 body[2][kWin];           // the frame's two symbol bodies in time (skewed windows)
    uint2 res[kMaxSnr];             // per SNR point of the current frame: {packed rail errors, sum |e|^2}, booked once per frame
};

// Replay of one (frame, SNR point) of the Monte-Carlo kernel in the reference's arithmetic (rare path of kArithChecked):
// the same Philox draws, exact channel, exact transform, exact decision stage.  txp3: the lane's three bit pairs,
// two bits each.  Returns {packed rail errors, lane's sum |e|^2}, not yet reduced over the warp.
__device__ __noinline__ uint2 mc_point_replay(const float2 *src, double sigma_d, uint32_t seed, uint32_t stream, uint64_t fr,
                                              uint32_t txp3, float2 *ws_tile, float2 *ws_lts, unsigned long long *replayed)
{
    const int lane = threadIdx.x & 31, grp = lane >> 3, u = lane & 7;
    Tw<true> tw; tw.load(u);
    const ItemConst ic = make_items(lane);
    const int blk_base = (grp < 2 ? 8 + 16 * grp : 44 + 20 * (grp - 2)) + u;
    float za[4], zb[4];
    philox_normals4(seed, stream, fr, (uint32_t)blk_base, kDomainNoise, za);
    philox_normals4(seed, stream, fr, (uint32_t)(blk_base + 8), kDomainNoise, zb);
    float2 r[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = slot_m<true>(i);
        float2 s = src[u + 8 * m];
        s.x = add_noise<true>(s.x, m < 4 ? za[m & 3] : zb[m & 3], sigma_d, 0.f);
        r[i] = s;
    }
    fft64<true>(r, tw, ws_tile + grp * kGroupPitch, u);
    float2 *dst = grp < 2 ? ws_lts + grp * kWin : ws_tile + (grp - 2) * kWin;
#pragma unroll
    for (int j = 0; j < 8; ++j) dst[u + 8 * j] = r[j];
    __syncwarp();
    float e2 = 0.f;
    uint32_t pk = 0;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const float2 A = ws_lts[ic.bin[t]], B = ws_lts[kWin + ic.bin[t]];
        const float2 Hh = make_float2(__fmul_rn(__fadd_rn(A.x, B.x), ic.sc[t]), __fmul_rn(__fadd_rn(A.y, B.y), ic.sc[t]));
        pk += item_eval<true>(ws_tile[ic.f_off[t]], Hh, ic.sc[t], (txp3 >> (2 * t)) & 3u, e2);
    }
    __syncwarp();
    if (lane == 0 && replayed != nullptr) atomicAdd(replayed, 1ull);
    return make_uint2(pk, __float_as_uint(e2));
}

// ARITH: kArithFast, kArithExact, or kArithChecked = exact transmitter, power and channel, receiver speculated in fp32
// with verified decisions and exact replay (see above) -- the totals of kArithExact.
// MP = true is configs[4] fused the same way: per-frame random taps (Philox domain 2, as k_multipath<true>) are applied
// to the whole 320-sample frame in shared memory (same operation order as k_multipath), the power is that of the faded
// frame (as frame_power() computes it), and the SNR loop runs on the faded windows.
struct MpWarp {
    float2 fx[320];                 // the transmitted frame, LTS || (CP + body) x 2
    float2 fw[4][kWin];             // faded LTS halves and symbol bodies (skewed windows)
    float2 sh[kMaxTaps];            // this frame's taps
};
template <bool MP> __host__ __device__ constexpr int mc_terms_per_warp() { return MP ? 320 : 160; }

template <int ARITH, bool MP = false>
__global__ void __launch_bounds__(kThreads, 2) k_mc_philox(McParams p)
{
    constexpr bool EXACT = ARITH == kArithExact;                // receiver arithmetic of the main path
    constexpr bool CHECKED = ARITH == kArithChecked;
    constexpr bool TX_EXACT = EXACT || CHECKED;                 // transmitter, power, channel
    // The fast Monte-Carlo kernels stay plain fp32: their results are statistical (no reference draws to match), and the EVM guard
    // of the fast receivers costs 12 % here (3.7 -> 3.3e9 symbols/s) -- the staged Philox route switches it off too (evm_guard = 0).
    constexpr bool SPEC = CHECKED;
    constexpr int LEVEL = 2;
    extern __shared__ __align__(128) unsigned char s_raw[];
    WarpShared *ws_all = reinterpret_cast<WarpShared *>(s_raw);
    float2 *s_ltsx = reinterpret_cast<float2 *>(s_raw + sizeof(WarpShared) * kWarpsPerBlock);   // [2][kWin] LTS halves, time
    double *s_terms = reinterpret_cast<double *>(s_ltsx + 2 * kWin);                            // [warps][160 | 320] (EXACT power)
    MpWarp *mp_all = reinterpret_cast<MpWarp *>(s_terms + kWarpsPerBlock * mc_terms_per_warp<MP>());

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, u = lane & 7;
    WarpShared &ws = ws_all[warp];
    float2 *tile = ws.tile + grp * kGroupPitch;
    Tw<EXACT> tw; tw.load(u);
    const ItemConst ic = make_items(lane);
    const float k4[3] = {4.f * ic.sc[0], 4.f * ic.sc[1], 4.f * ic.sc[2]};     // 1 / sc (CHECKED)
    int dmap_tx[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) dmap_tx[i] = c_tab.bin_data[8 * slot_m<TX_EXACT>(i) + u];

    for (int i = threadIdx.x; i < 128; i += kThreads) s_ltsx[(i >> 6) * kWin + (i & 63)] = c_tab.lts_time[32 + i];
    if (MP) {                                                    // the LTS slot of the frame never changes
        MpWarp &mw = mp_all[warp];
        for (int i = lane; i < 160; i += 32) mw.fx[i] = c_tab.lts_time[i];
    }
    __syncthreads();

    const float2 *src = MP ? mp_all[warp].fw[grp] : (grp < 2 ? s_ltsx + grp * kWin : ws.body[grp - 2]);
    const int blk_base = (grp < 2 ? 8 + 16 * grp : 44 + 20 * (grp - 2)) + u;        // window_block_base(n0) + u
    const double q = (double)kQpsk;
    const float inv_ref2 = (float)(1.0 / (96.0 * (2.0 * q * q)));
    // Per-SNR totals live in registers: lane L owns SNR points L and L + 32 (n_snr <= 64).  The float EVM sums are
    // flushed into doubles every 64 frames.
    uint32_t m_i[2] = {0, 0}, m_q[2] = {0, 0}, m_b[2] = {0, 0}, m_ferr[2] = {0, 0};
    float m_e2[2] = {0.f, 0.f}, m_evm[2] = {0.f, 0.f};
    double d_e2[2] = {0.0, 0.0}, d_evm[2] = {0.0, 0.0};
    uint32_t n_done = 0;

    for (long f = (long)blockIdx.x * kWarpsPerBlock + warp; f < p.n_frames; f += (long)gridDim.x * kWarpsPerBlock) {
        const uint64_t fr = p.frame0 + (uint64_t)f;
        // ---- payload bits (Philox, one block per symbol) and Transmitter :500-565 for the two symbols
        const uint4 b0 = Philox::run(make_uint4((uint32_t)fr, (uint32_t)(fr >> 32), 0u, kDomainBits), p.seed, 0u);
        const uint4 b1 = Philox::run(make_uint4((uint32_t)fr, (uint32_t)(fr >> 32), 1u, kDomainBits), p.seed, 0u);
        // the lane's three bit pairs of this frame (constant over the SNR loop)
        uint32_t txp[3];
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            const int wsel = ic.word[t];
            const uint32_t w = wsel == 0 ? b0.x : wsel == 1 ? b0.y : wsel == 2 ? b0.z : wsel == 3 ? b1.x : wsel == 4 ? b1.y : b1.z;
            txp[t] = w >> ic.shift[t];
        }
        float P;
        {
            const bool s1 = (grp & 1) != 0;
            const uint32_t w0 = s1 ? b1.x : b0.x, w1 = s1 ? b1.y : b0.y, w2 = s1 ? b1.z : b0.z;
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
            if constexpr (CHECKED) {                              // the exact twiddles live only here: once per frame
                Tw<true> twx; twx.load(u);
                fft64<true>(v, twx, tile, u);
            } else {
                fft64<EXACT>(v, tw, tile, u);
            }
            float pw = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int np = u + 8 * ((j + 4) & 7);
                const float2 y = make_float2(v[j].x * 0.015625f, -v[j].y * 0.015625f);
                if (MP) {
                    if (grp >= 2) {
                        float2 *sym = mp_all[warp].fx + 160 + 80 * (grp - 2);
                        sym[16 + np] = y;
                        if (np >= 48) sym[np - 48] = y;                 // cyclic prefix :559-565
                    }
                } else {
                    if (grp >= 2) ws.body[grp - 2][np] = y;
                    const float e = fmaf(y.x, y.x, y.y * y.y);
                    pw += (grp >= 2) ? (np >= 48 ? 2.f * e : e) : 0.f;  // the CP repeats samples 48..63
                }
            }
            __syncwarp();
            if (MP) {
                MpWarp &mw = mp_all[warp];
                const int n_taps = p.n_taps;
                if (2 * lane < n_taps) {                                // taps of this frame: k_multipath<true>
                    const float scale = sqrtf(0.5f / (float)n_taps);
                    float z[4];
                    philox_normals4(p.seed, 0u, fr, (uint32_t)lane, kDomainTaps, z);
                    mw.sh[2 * lane] = make_float2(scale * z[0], scale * z[1]);
                    if (2 * lane + 1 < n_taps) mw.sh[2 * lane + 1] = make_float2(scale * z[2], scale * z[3]);
                }
                __syncwarp();
                double *terms = s_terms + warp * 320;
                for (int n = lane; n < 320; n += 32) {                   // y[n] = sum_l h[l] x[n-l], descending l, no FMA
                    float ar = 0.f, ai = 0.f;
                    for (int l = (n_taps - 1 < n ? n_taps - 1 : n); l >= 0; --l) {
                        const float2 a = mw.fx[n - l], b = mw.sh[l];
                        ar = __fadd_rn(ar, __fsub_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)));
                        ai = __fadd_rn(ai, __fadd_rn(__fmul_rn(a.x, b.y), __fmul_rn(a.y, b.x)));
                    }
                    // the windows the receiver reads: 32..95, 96..159, 176..239, 256..319
                    const int w = n < 160 ? (n >= 32 ? (n - 32) >> 6 : -1) : ((n - 160) % 80 >= 16 ? 2 + (n - 160) / 80 : -1);
                    if (w >= 0) mw.fw[w][w < 2 ? (n - 32) & 63 : (n - 160) % 80 - 16] = make_float2(ar, ai);
                    if (TX_EXACT) { const double h = hypot_glibc((double)ar, (double)ai); terms[n] = __dmul_rn(h, h); }
                    else pw = fmaf(ar, ar, fmaf(ai, ai, pw));            // k_frame_power_fast's order
                }
                __syncwarp();
                if (TX_EXACT) {                                          // frame_power(): the whole faded frame, in order
                    float acc = 0.f;
                    if (lane == 0) for (int i = 0; i < 320; ++i) acc = __double2float_rn(__dadd_rn((double)acc, terms[i]));
                    P = __fdiv_rn(__shfl_sync(0xffffffffu, acc, 0), 320.f);
                } else {
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) pw += __shfl_xor_sync(0xffffffffu, pw, o);
                    P = pw / 320.f;
                }
            } else if (TX_EXACT) {
                // OFDM.c:637-643 on the 320-sample frame: the LTS prefix is a constant, the 160 data samples follow in order
                double *terms = s_terms + warp * 160;
                for (int i = lane; i < 160; i += 32) {
                    const int s = i / 80, k = i - 80 * s;
                    const float2 y = ws.body[s][k < 16 ? 48 + k : k - 16];
                    const double h = hypot_glibc((double)y.x, (double)y.y);
                    terms[i] = __dmul_rn(h, h);
                }
                __syncwarp();
                float acc = c_tab.lts_power_prefix;
                if (lane == 0) for (int i = 0; i < 160; ++i) acc = __double2float_rn(__dadd_rn((double)acc, terms[i]));
                P = __fdiv_rn(__shfl_sync(0xffffffffu, acc, 0), 320.f);
            } else {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) pw += __shfl_xor_sync(0xffffffffu, pw, o);
                P = (pw + c_tab.lts_power_sum) * (1.f / 320.f);
            }
        }
        float sqrtP;
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sqrtP) : "f"(P));
        // ---- SNR loop OFDM.c:1202: channel :635 + receiver :1018-1165 on the frame held in shared memory
        // exact noise scale sqrt((double)(P / snr)) (:647, :651) of every SNR point, one (two) per lane, once per frame
        double sig_lo = 0.0, sig_hi = 0.0;
        if (TX_EXACT) {
            if (lane < p.n_snr) sig_lo = __dsqrt_rn((double)__fdiv_rn(P, p.snr_lin[lane]));
            if (lane + 32 < p.n_snr) sig_hi = __dsqrt_rn((double)__fdiv_rn(P, p.snr_lin[lane + 32]));
        }
        // The warp sums of a point (one REDUX, five dependent shuffles) are finished one iteration late, on top of the next
        // point's Philox rounds, and the owner lanes book all points of the frame at once from ws.res (no per-point branch).
        uint32_t pk_pend = 0;
        float e2_pend = 0.f;
        for (int si = 0; si < p.n_snr; ++si) {
            {
                float rs = e2_pend;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, o);
                if (lane == 0 && si > 0) ws.res[si - 1] = make_uint2(pk_pend, __float_as_uint(rs));
            }
            double sigma_d = 0.0; float sigma_f;
            if (TX_EXACT) {
                sigma_d = __shfl_sync(0xffffffffu, si < 32 ? sig_lo : sig_hi, si & 31);
                sigma_f = (float)sigma_d;
                if (EXACT) sigma_d = __dmul_rn(sigma_d, kTwScale);          // add_noise_s (the all-exact kernel is XU-bound)
            } else { sigma_f = sqrtP * p.inv_sqrt_snr[si]; sigma_d = (double)sigma_f; }      // (the replay of a guarded bin uses the same scale)
            float za[4], zb[4];
            const uint32_t stream = p.stream[si];
            philox_normals4(p.seed, stream, fr, (uint32_t)blk_base, kDomainNoise, za);
            philox_normals4(p.seed, stream, fr, (uint32_t)(blk_base + 8), kDomainNoise, zb);
            float2 r[8];
            float2 n2 = make_float2(0.f, 0.f);                    // CHECKED: the lane's share of the window's energy (re^2, im^2)
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int m = slot_m<EXACT>(i);
                float2 s = src[u + 8 * m];
                const float z = m < 4 ? za[m & 3] : zb[m & 3];
                if (SPEC) { s.x = fmaf(sigma_f, z, s.x); n2 = __ffma2_rn(s, s, n2); }         // speculated channel (see kChanRadius)
                else s.x = add_noise_s<EXACT>(s.x, z, sigma_d, sigma_f);
                r[i] = s;
            }
            fft64<EXACT>(r, tw, tile, u);
            // exchange: LTS groups publish A / B, data groups publish F (the transform tile is free now)
            float2 *dst = grp < 2 ? ws.lts[grp] : ws.tile + (grp - 2) * kWin;
#pragma unroll
            for (int j = 0; j < 8; ++j) dst[u + 8 * j] = r[j];
            float rad = 0.f;
            if (SPEC) rad = window_radius(n2, p.radius_scale, p.radius_chan * sqrtP);
            __syncwarp();
            float e2 = 0.f;
            uint32_t pk = 0;
            if (SPEC) {
                float2 e2v = make_float2(0.f, 0.f);
                const float rA = __shfl_sync(0xffffffffu, rad, 0), rB = __shfl_sync(0xffffffffu, rad, 8);
                const float r0 = __shfl_sync(0xffffffffu, rad, 16), r1 = __shfl_sync(0xffffffffu, rad, 24);
                const float rH2 = rA + rB;                                        // 2 r_H
                const float den_min4 = (p.evm_guard * rH2) * (p.evm_guard * rH2);
                bool doubt = false;
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const float2 A = ws.lts[0][ic.bin[t]], B = ws.lts[1][ic.bin[t]];
                    const float2 G = cadd(A, B);
                    const float rF = ic.f_off[t] < kWin ? r0 : r1;
                    pk += process_bin_spec<LEVEL>(ws.tile[ic.f_off[t]], G, k4[t], txp[t], rF, rH2, den_min4, e2v, doubt);
                }
                e2 = e2v.x + e2v.y;
                __syncwarp();
                if (__any_sync(0xffffffffu, doubt)) {             // not provably the reference's decisions / EVM: replay exactly
                    const uint32_t txp3 = (txp[0] & 3u) | ((txp[1] & 3u) << 2) | ((txp[2] & 3u) << 4);
                    const uint2 rr = mc_point_replay(src, sigma_d, p.seed, stream, fr, txp3, ws.tile, &ws.lts[0][0], p.replayed);
                    pk = rr.x; e2 = __uint_as_float(rr.y);
                }
            } else {
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const float2 A = ws.lts[0][ic.bin[t]], B = ws.lts[1][ic.bin[t]];
                    const float2 Hh = make_float2(__fmul_rn(__fadd_rn(A.x, B.x), ic.sc[t]), __fmul_rn(__fadd_rn(A.y, B.y), ic.sc[t]));
                    pk += item_eval<EXACT>(ws.tile[ic.f_off[t]], Hh, ic.sc[t], txp[t], e2);
                }
                __syncwarp();
            }
            pk_pend = __reduce_add_sync(0xffffffffu, pk);           // one REDUX: the three 8-bit fields stay below 97
            e2_pend = e2;
        }
        {
            float rs = e2_pend;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, o);
            if (lane == 0) ws.res[p.n_snr - 1] = make_uint2(pk_pend, __float_as_uint(rs));
        }
        __syncwarp();
        // the lane that owns an SNR point books the frame's result for it (lanes beyond n_snr read stale words and add nothing)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint2 rr = ws.res[lane + 32 * h];
            const bool mine = lane + 32 * h < p.n_snr;
            const uint32_t pkh = mine ? rr.x : 0u;
            const float e2h = mine ? __uint_as_float(rr.y) : 0.f;
            float evm;
            asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(evm) : "f"(e2h * inv_ref2));                // :1124
            m_i[h] += pkh & 0xFFu; m_q[h] += (pkh >> 8) & 0xFFu; m_b[h] += pkh >> 16; m_ferr[h] += pkh != 0u;
            m_e2[h] += e2h; m_evm[h] += evm;
        }
        __syncwarp();
        n_done += 1;
        if ((n_done & 63u) == 0u) {
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

inline size_t mc_smem_bytes(bool multipath = false)
{
    return sizeof(WarpShared) * kWarpsPerBlock + 2 * kWin * sizeof(float2) + kWarpsPerBlock * (multipath ? 320 : 160) * sizeof(double) +
           (multipath ? sizeof(MpWarp) * kWarpsPerBlock : 0);
}

// payload bits of the Philox bit stream, for callers that want the same frames in HBM (symbol s = block s)
__global__ void k_philox_bits(uint32_t seed, uint64_t frame0, long n_symbols, int n_sym, uint32_t *__restrict__ bits)
{
    long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_symbols) return;
    const long f = t / n_sym; const uint32_t s = (uint32_t)(t - f * n_sym);
    const uint64_t fr = frame0 + (uint64_t)f;
    const uint4 r = Philox::run(make_uint4((uint32_t)fr, (uint32_t)(fr >> 32), s, kDomainBits), seed, 0u);
    bits[t * 3] = r.x; bits[t * 3 + 1] = r.y; bits[t * 3 + 2] = r.z;
}


// ------------------------------------------------------------------------------------------------
// k_stream_rx2 -- channel + receiver for HBM-resident frames (n_sym = 2), TMA-staged.
//
// Each warp streams its frames through a private ring of shared-memory stages.  One lane issues bulk
// async copies (cp.async.bulk, the TMA engine's 1-D mode; SASS UBLKCP) for exactly the samples the receiver
// uses -- the two LTS halves and the two symbol bodies of the IQ frame and, for injected noise, of the draw
// buffer -- straight into bank-skewed windows, and arms an mbarrier with the byte count; the warp waits
// on the barrier's phase, pulls its samples into registers, and immediately re-arms the stage for the frame
// two iterations ahead, so HBM latency is covered by a full frame of transform work without holding
// any prefetch registers.
namespace tma {
__device__ __forceinline__ uint32_t saddr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(saddr(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(saddr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(saddr(dst)), "l"(src), "r"(bytes), "r"(saddr(bar)) : "memory");
}
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void expect_tx_addr(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_addr(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void wait_addr(uint32_t bar_saddr, uint32_t phase)
{
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "LAB_WAIT:\n"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
                 "@p bra DONE;\n"
                 "bra LAB_WAIT;\n"
                 "DONE:\n"
                 "}" ::"r"(bar_saddr), "r"(phase) : "memory");
}
__device__ __forceinline__ void wait(uint64_t *bar, uint32_t phase)
{
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "LAB_WAIT:\n"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
                 "@p bra DONE;\n"
                 "bra LAB_WAIT;\n"
                 "DONE:\n"
                 "}" ::"r"(saddr(bar)), "r"(phase) : "memory");
}
}  // namespace tma

// ------------------------------------------------------------------------------------------------
// k_tx_frames2 -- the transmitter for the default frame shape (LTS + 2 symbols), frames leaving through the TMA engine.
// A warp builds two frames per pass (lane group 2 s + k = symbol s of frame k) in shared memory -- the LTS slot is a
// constant of the build and is written into the frame images once, at kernel start -- and one elected lane hands each
// finished 2560-byte frame image to a bulk async copy (cp.async.bulk.global.shared::cta, SASS UBLKCP): the SM issues two
// store instructions per pair of frames instead of ~60 per lane, and HBM sees whole, aligned 2560-byte writes.  Two sets of
// images alternate so that a pass can fill one while the copy engine drains the other (bulk_group / wait_group.read).
// The image of the second frame sits 8 elements further (pitch 328) so that the two half-warp partners never hit the
// same bank pair.
constexpr int kTxPitch = 328;           // float2 per frame image: 320 + 8 of skew
struct alignas(16) TxWarp { float2 img[2][2][kTxPitch]; };
inline size_t tx2_smem_bytes() { return sizeof(TxWarp) * kWarpsPerBlock; }

namespace tma {
__device__ __forceinline__ void bulk_s2g(void *dst_global, uint32_t src_shared, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_global), "r"(src_shared), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
}  // namespace tma

template <bool EXACT>
__global__ void __launch_bounds__(kThreads) k_tx_frames2(const uint32_t *__restrict__ bits, float2 *__restrict__ frames, long n_frames)
{
    __shared__ float2 s_tile[kWarpsPerBlock][kWarpTile];
    extern __shared__ __align__(128) unsigned char s_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, u = lane & 7;
    TxWarp &tw_s = reinterpret_cast<TxWarp *>(s_raw)[warp];
    float2 *tile = s_tile[warp] + grp * kGroupPitch;
    Tw<EXACT> tw; tw.load(u);
    int dmap[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) dmap[i] = c_tab.bin_data[8 * slot_m<EXACT>(i) + u];   // input index n <-> centred (n+32)%64
    for (int i = lane; i < 4 * 160; i += 32) tw_s.img[i / 320][(i / 160) & 1][i % 160] = c_tab.lts_time[i % 160];      // LTS slot :573
    __syncwarp();
    const int k = grp & 1, sy = grp >> 1;                        // frame of the pair, symbol of the frame (half-warp partners: the two frames)
    const long n_pairs = (n_frames + 1) / 2;
    const long pr_step = (long)gridDim.x * kWarpsPerBlock;
    uint32_t it = 0;
    // the payload words of a pass are fetched one pass ahead: they are the first thing a pass needs, and with two resident blocks
    // per SM (the exact arithmetic's 96 registers) nothing else covered their latency (ncu: long_scoreboard 2.0 per issue)
    // (the fp32 build runs four blocks per SM at 63 registers and is faster without the three extra registers: 0.92 vs 0.87 of peak)
    uint32_t nw0 = 0, nw1 = 0, nw2 = 0;
    if (EXACT) {
        const long f = 2 * ((long)blockIdx.x * kWarpsPerBlock + warp) + k;
        if (f < n_frames) { const uint32_t *w = bits + (f * 2 + sy) * 3; nw0 = w[0]; nw1 = w[1]; nw2 = w[2]; }
    }
    for (long pr = (long)blockIdx.x * kWarpsPerBlock + warp; pr < n_pairs; pr += pr_step, ++it) {
        const int st = (int)(it & 1u);
        const long f = 2 * pr + k;
        uint32_t w0 = nw0, w1 = nw1, w2 = nw2;
        if (EXACT) {
            const long fn = f + 2 * pr_step;
            nw0 = nw1 = nw2 = 0;
            if (fn < n_frames) { const uint32_t *w = bits + (fn * 2 + sy) * 3; nw0 = w[0]; nw1 = w[1]; nw2 = w[2]; }
        } else if (f < n_frames) { const uint32_t *w = bits + (f * 2 + sy) * 3; w0 = w[0]; w1 = w[1]; w2 = w[2]; }
        float2 v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            // grid value at centred index (n+32)%64 (ifft_shift :208), conjugated (:328)
            const int d = dmap[i];
            float2 x = make_float2(0.f, -0.f);
            if (d >= 0) { x = qpsk_point(bit_pair(w0, w1, w2, d)); x.y = -x.y; }
            else if (d == -2) x.x = 1.f;
            else if (d == -3) x.x = -1.f;
            v[i] = x;
        }
        fft64<EXACT>(v, tw, tile, u);
        // the image set `st` was handed to the copy engine two passes ago: it must have been read before it is overwritten
        if (lane == 0) tma::bulk_wait_read<1>();
        __syncwarp();
        float2 *dst = tw_s.img[st][k] + 160 + 80 * sy;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int np = u + 8 * ((j + 4) & 7);               // fft_shift inside ifft's fft() -> 32-sample rotation (Q4)
            const float2 y = make_float2(v[j].x * 0.015625f, -v[j].y * 0.015625f);
            dst[16 + np] = y;                                   // body :564
            if (np >= 48) dst[np - 48] = y;                     // CP   :563
        }
        tma::fence_proxy_async();                               // generic-proxy writes -> visible to the async proxy
        __syncwarp();
        if (lane == 0) {
            tma::bulk_s2g(frames + (2 * pr) * 320, tma::saddr(tw_s.img[st][0]), 2560);
            if (2 * pr + 1 < n_frames) tma::bulk_s2g(frames + (2 * pr + 1) * 320, tma::saddr(tw_s.img[st][1]), 2560);
            tma::bulk_commit();
        }
    }
    if (lane == 0) tma::bulk_wait_read<0>();                    // shared memory must outlive the copies that read it
}

constexpr int kStages = 2;          // the ring indexing below (k & 1, k >> 1) relies on it

template <bool WITH_DRAWS> struct alignas(16) StreamStage {     // bulk-copy destinations must be 16-byte aligned
    float2 x[4][kWin];              // LTS1, LTS2, sym0 body, sym1 body (skewed windows)
    float g[4][kWin];               // the matching draws (injected noise only)
};
template <> struct alignas(16) StreamStage<false> {
    float2 x[4][kWin];
    float g[1][4];                  // never touched
};
template <bool WITH_DRAWS> struct alignas(16) StreamWarp {
    float2 tile[kWarpTile];
    float2 lts[2][kWin];
    StreamStage<WITH_DRAWS> st[kStages];
    uint64_t bar[kStages];
    float radius[4];                // kArithChecked: error radius of each window's transform (see below)
};
// Replay of one frame in the reference's arithmetic (rare path of kArithChecked): samples straight from global
// memory, exact channel, exact transform, exact decision stage.  Returns {packed rail errors, lane's sum |e|^2}.
template <int NOISE>
__device__ __noinline__ uint2 stream_frame_replay(const float2 *frame, const float *draws, const uint32_t *wb, double sigma_d,
                                                  uint32_t seed, uint32_t stream, uint64_t frame_id, float2 *ws_tile, float2 *ws_lts,
                                                  unsigned long long *replayed)
{
    const int lane = threadIdx.x & 31, grp = lane >> 3, u = lane & 7;
    Tw<true> tw; tw.load(u);
    const ItemConst ic = make_items(lane);
    const int n0 = grp == 0 ? 32 : grp == 1 ? 96 : grp == 2 ? 176 : 256;
    float z[8];
    if (NOISE == kNoisePhilox) {                                  // the same draws as the speculated pass (window block layout)
        const int blk_base = (grp < 2 ? 8 + 16 * grp : 44 + 20 * (grp - 2)) + u;
        float za[4], zb[4];
        philox_normals4(seed, stream, frame_id, (uint32_t)blk_base, kDomainNoise, za);
        philox_normals4(seed, stream, frame_id, (uint32_t)(blk_base + 8), kDomainNoise, zb);
#pragma unroll
        for (int m = 0; m < 4; ++m) { z[m] = za[m]; z[4 + m] = zb[m]; }
    }
    float2 v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = slot_m<true>(i), n = n0 + u + 8 * m;
        float2 smp = frame[n];
        if (NOISE == kNoiseInject) smp.x = add_noise<true>(smp.x, draws[n], sigma_d, 0.f);
        if (NOISE == kNoisePhilox) smp.x = add_noise<true>(smp.x, z[m], sigma_d, 0.f);
        v[i] = smp;
    }
    fft64<true>(v, tw, ws_tile + grp * kGroupPitch, u);
    float2 *dst = grp < 2 ? ws_lts + grp * kWin : ws_tile + (grp - 2) * kWin;
#pragma unroll
    for (int j = 0; j < 8; ++j) dst[u + 8 * j] = v[j];
    __syncwarp();
    float e2 = 0.f;
    uint32_t pk = 0;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const float2 A = ws_lts[ic.bin[t]], B = ws_lts[kWin + ic.bin[t]];
        const float2 Hh = make_float2(__fmul_rn(__fadd_rn(A.x, B.x), ic.sc[t]), __fmul_rn(__fadd_rn(A.y, B.y), ic.sc[t]));   // :848
        pk += item_eval<true>(ws_tile[ic.f_off[t]], Hh, ic.sc[t], wb[ic.word[t]] >> ic.shift[t], e2);
    }
    __syncwarp();
    if (lane == 0 && replayed != nullptr) atomicAdd(replayed, 1ull);
    return make_uint2(pk, __float_as_uint(e2));
}

// resident blocks per SM the launch bounds ask for.  Round 1 ran the fp32 kernels without injected draws at three (80 registers);
// with the EVM guard and its replay call they need more than 80 registers (spills made three blocks 2x slower than two).
static_assert(sizeof(StreamStage<false>) % 16 == 0 && sizeof(StreamStage<true>) % 16 == 0 && sizeof(StreamWarp<false>) % 16 == 0, "stage alignment");
#ifndef OFDM_FAST_STREAM_BLOCKS
#define OFDM_FAST_STREAM_BLOCKS 2       // A/B knob (tools/ab.sh): resident blocks per SM of the fast kernels without injected draws
#endif
template <int ARITH, int NOISE> constexpr int stream_blocks_per_sm() { return (ARITH == kArithFast && NOISE != kNoiseInject) ? OFDM_FAST_STREAM_BLOCKS : 2; }

template <int ARITH, int NOISE>
__global__ void __launch_bounds__(kThreads, stream_blocks_per_sm<ARITH, NOISE>()) k_stream_rx2(RxParams p)
{
    constexpr bool EXACT = ARITH == kArithExact;                // transform / decision arithmetic of the main path
    constexpr bool CHECKED = ARITH == kArithChecked;
    constexpr bool SPEC = ARITH != kArithExact;                 // fp32 speculation + exact replay: every rail decision verified (checked) or the EVM guard only (fast)
    constexpr int LEVEL = CHECKED ? 2 : 1;
    extern __shared__ __align__(128) unsigned char s_raw[];
    __shared__ unsigned long long s_cnt[kWarpsPerBlock][4];
    __shared__ double s_sum[kWarpsPerBlock][2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, u = lane & 7;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);                  // same value, provably warp-uniform
    using SW = StreamWarp<NOISE == kNoiseInject>;
    using SS = StreamStage<NOISE == kNoiseInject>;
    SW &ws = reinterpret_cast<SW *>(s_raw)[warp];
    SW &ws_u = reinterpret_cast<SW *>(s_raw)[warp_u];
    float2 *tile = ws.tile + grp * kGroupPitch;
    Tw<EXACT> tw; tw.load(u);
    const ItemConst ic = make_items(lane);
    const float k4[3] = {4.f * ic.sc[0], 4.f * ic.sc[1], 4.f * ic.sc[2]};     // 1 / sc (CHECKED)
    constexpr int len = 320;
    const long stride = (long)gridDim.x * kWarpsPerBlock;
    const long f_first = (long)blockIdx.x * kWarpsPerBlock + warp_u;
    const double q = (double)kQpsk;
    const double ref2_frame = 96.0 * (2.0 * q * q);
    const float inv_ref2 = (float)(1.0 / ref2_frame);
    constexpr uint32_t kBytes = 4 * 512 + (NOISE == kNoiseInject ? 4 * 256 : 0);

    // A stage refill = one expect_tx + four (eight with draws) bulk copies, issued by one elected lane.  UBLKCP takes
    // uniform-register operands, so every operand is derived from warp-uniform values (the warp index is
    // broadcast with a shuffle so that the compiler can prove it) and stays on the uniform datapath.
    const uint32_t stage0 = tma::saddr(&ws_u.st[0]);
    const uint32_t bar0 = tma::saddr(&ws_u.bar[0]);
    auto issue = [&](long f, int s) {          // f, s warp-uniform; whole warp calls
        if (tma::elect_one()) {
            const uint32_t bar = bar0 + 8u * (uint32_t)s;
            const uint32_t dst = stage0 + (uint32_t)s * (uint32_t)sizeof(SS);
            const char *x = reinterpret_cast<const char *>(p.in) + f * (len * 8);
            tma::expect_tx_addr(bar, kBytes);
            tma::bulk_addr(dst + 0 * kWin * 8, x + 32 * 8, 512, bar);             // Channel_Estimation :837
            tma::bulk_addr(dst + 1 * kWin * 8, x + 96 * 8, 512, bar);             //                    :838
            tma::bulk_addr(dst + 2 * kWin * 8, x + 176 * 8, 512, bar);            // CP strip :1028, symbol 0
            tma::bulk_addr(dst + 3 * kWin * 8, x + 256 * 8, 512, bar);            //                 symbol 1
            if (NOISE == kNoiseInject) {
                const char *g = reinterpret_cast<const char *>(p.g) + f * (len * 4);
                const uint32_t gd = dst + 4 * kWin * 8;
                tma::bulk_addr(gd + 0 * kWin * 4, g + 32 * 4, 256, bar);
                tma::bulk_addr(gd + 1 * kWin * 4, g + 96 * 4, 256, bar);
                tma::bulk_addr(gd + 2 * kWin * 4, g + 176 * 4, 256, bar);
                tma::bulk_addr(gd + 3 * kWin * 4, g + 256 * 4, 256, bar);
            }
        }
    };

    if (lane == 0) {
        for (int s = 0; s < kStages; ++s) tma::mbar_init(&ws.bar[s], 1);
        tma::fence_mbar_init();
    }
    __syncwarp();
    for (int s = 0; s < kStages; ++s)
        if (f_first + s * stride < p.n_frames) issue(f_first + s * stride, s);

    uint32_t a_i = 0, a_q = 0, a_both = 0, a_ferr = 0, a_frames = 0;
    double a_e2 = 0.0, a_evm = 0.0;
    const int blk_base = (grp < 2 ? 8 + 16 * grp : 44 + 20 * (grp - 2)) + u;
    uint32_t k = 0;                                   // frames this warp has consumed (ring position)
    for (long f_chunk = f_first; f_chunk < p.n_frames; f_chunk += 32 * stride) {
        double sig_mine = 0.0;
        if (NOISE != kNoiseNone) {
            const long fl = f_chunk + lane * stride;
            if (fl < p.n_frames) sig_mine = __dsqrt_rn((double)__fdiv_rn(p.power[fl], p.snr_lin));   // :647, :651
        }
        float c_e2 = 0.f, c_evm = 0.f;
        for (int kk = 0; kk < 32; ++kk, ++k) {
            const long f = f_chunk + kk * stride;
            if (f >= p.n_frames) break;
            const int s = (int)(k & 1u);
            const uint32_t phase = (k >> 1) & 1u;
            const double sigma_d = NOISE != kNoiseNone ? __shfl_sync(0xffffffffu, sig_mine, kk) : 0.0;
            const float sigma_f = (float)sigma_d;
            const double sigma_s = __dmul_rn(sigma_d, kTwScale);        // for add_noise_s
            // this frame's payload words for the lane's three items (used after the transform)
            const uint32_t *wb = p.tx_bits + f * 6;
            const uint32_t w0 = wb[ic.word[0]], w1 = wb[ic.word[1]], w2 = wb[ic.word[2]];
            float z[8];
            if (NOISE == kNoisePhilox) {
                float za[4], zb[4];
                philox_normals4(p.seed, p.stream, p.frame0 + (uint64_t)f, (uint32_t)blk_base, kDomainNoise, za);
                philox_normals4(p.seed, p.stream, p.frame0 + (uint64_t)f, (uint32_t)(blk_base + 8), kDomainNoise, zb);
#pragma unroll
                for (int m = 0; m < 4; ++m) { z[m] = za[m]; z[4 + m] = zb[m]; }
            }
            tma::wait_addr(bar0 + 8u * (uint32_t)s, phase);
            float2 v[8];
            float2 n2 = make_float2(0.f, 0.f);                    // CHECKED: the lane's share of the window's energy (re^2, im^2)
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int m = slot_m<EXACT>(i);
                float2 smp = ws.st[s].x[grp][u + 8 * m];
                if (NOISE == kNoiseInject) smp.x = add_noise<EXACT>(smp.x, ws.st[s].g[grp][u + 8 * m], sigma_d, sigma_f);   // CHECKED: speculated (kChanRadius)
                if (NOISE == kNoisePhilox) smp.x = add_noise<EXACT>(smp.x, z[m], sigma_d, sigma_f);
                if (SPEC) n2 = __ffma2_rn(smp, smp, n2);
                v[i] = smp;
            }
            __syncwarp();                                         // every lane has its samples: the stage can be refilled
            if (f + kStages * stride < p.n_frames) issue(f + kStages * stride, s);
            fft64<EXACT>(v, tw, tile, u);
            float2 *dst = grp < 2 ? ws.lts[grp] : ws.tile + (grp - 2) * kWin;
#pragma unroll
            for (int j = 0; j < 8; ++j) dst[u + 8 * j] = v[j];
            if (SPEC) {
                const float r = window_radius(n2, p.radius_scale, NOISE != kNoiseNone ? p.radius_chan * sigma_f : 0.f);
                if (u == 0) ws.radius[grp] = r;
            }
            __syncwarp();
            float f_e2 = 0.f;
            uint32_t pk = 0;
            if (SPEC) {
                float2 e2v = make_float2(0.f, 0.f);
                const float4 rad = *reinterpret_cast<const float4 *>(ws.radius);
                const float rH2 = rad.x + rad.y;                                  // 2 r_H
                const float den_min4 = (p.evm_guard * rH2) * (p.evm_guard * rH2);
                bool doubt = false;
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const float2 A = ws.lts[0][ic.bin[t]], B = ws.lts[1][ic.bin[t]];
                    const float2 G = cadd(A, B);
                    const uint32_t w = t == 0 ? w0 : t == 1 ? w1 : w2;
                    const float rF = ic.f_off[t] < kWin ? rad.z : rad.w;               // the item's symbol
                    pk += process_bin_spec<LEVEL>(ws.tile[ic.f_off[t]], G, k4[t], w >> ic.shift[t], rF, rH2, den_min4, e2v, doubt);
                }
                f_e2 = e2v.x + e2v.y;
                __syncwarp();
                if (__any_sync(0xffffffffu, doubt)) {             // not provably the reference's decisions: replay exactly
                    const uint2 r = stream_frame_replay<NOISE>(p.in + f * len, NOISE == kNoiseInject ? p.g + f * len : nullptr,
                                                               p.tx_bits + f * 6, sigma_d, p.seed, p.stream, p.frame0 + (uint64_t)f,
                                                               ws.tile, &ws.lts[0][0], p.replayed);
                    pk = r.x; f_e2 = __uint_as_float(r.y);
                }
            } else {
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const float2 A = ws.lts[0][ic.bin[t]], B = ws.lts[1][ic.bin[t]];
                    const float2 Hh = make_float2(__fmul_rn(__fadd_rn(A.x, B.x), ic.sc[t]), __fmul_rn(__fadd_rn(A.y, B.y), ic.sc[t]));   // :848
                    const uint32_t w = t == 0 ? w0 : t == 1 ? w1 : w2;
                    pk += item_eval<EXACT>(ws.tile[ic.f_off[t]], Hh, ic.sc[t], w >> ic.shift[t], f_e2);
                }
                __syncwarp();
            }
            const bool any_err = __any_sync(0xffffffffu, pk != 0u);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) f_e2 += __shfl_xor_sync(0xffffffffu, f_e2, o);
            float evm;
            asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(evm) : "f"(f_e2 * inv_ref2));                                              // :1124
            a_i += pk & 0xFFu; a_q += (pk >> 8) & 0xFFu; a_both += pk >> 16;
            a_ferr += any_err; a_frames += 1;
            c_e2 += f_e2; c_evm += evm;
        }
        a_e2 += (double)c_e2; a_evm += (double)c_evm;
    }
    if (p.counters == nullptr) return;
    const uint32_t t_i = warp_sum(a_i), t_q = warp_sum(a_q), t_both = warp_sum(a_both);
    if (lane == 0) {
        s_cnt[warp][0] = (unsigned long long)t_i + 2ull * t_q - 2ull * t_both;     // bit errors (map of :423-430)
        s_cnt[warp][1] = (unsigned long long)t_i + t_q;
        s_cnt[warp][2] = a_ferr; s_cnt[warp][3] = a_frames;
        s_sum[warp][0] = a_e2; s_sum[warp][1] = a_evm;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long c[4] = {0, 0, 0, 0}; double sm[2] = {0, 0};
        for (int w = 0; w < kWarpsPerBlock; ++w) {
            for (int i = 0; i < 4; ++i) c[i] += s_cnt[w][i];
            for (int i = 0; i < 2; ++i) sm[i] += s_sum[w][i];
        }
        if (c[3] != 0) {
            ofdm_counters *o = p.counters;
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->bit_errors), c[0]);
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->rail_errors), c[1]);
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->frames_in_error), c[2]);
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->frames), c[3]);
            atomicAdd(reinterpret_cast<unsigned long long *>(&o->bits), c[3] * 192ull);
            atomicAdd(&o->sum_err2, sm[0]);
            atomicAdd(&o->sum_ref2, (double)c[3] * ref2_frame);
            atomicAdd(&o->sum_evm_lin, sm[1]);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// The streaming receiver for any number of data symbols.  A frame is a sequence of passes through the same ring:
// pass 0 = {LTS half 1, LTS half 2, symbol 0, symbol 1} exactly as k_stream_rx2, then four symbols per pass against the
// channel estimate left in shared memory by pass 0, their 192 data bins dealt out six per lane.  kArithChecked marks a frame whose
// decisions are not all provably the reference's and replays it whole (sweep_frame_replay) after its last pass.
struct SweepLane {                  // per-lane constants for the natural bins u + 8j
    uint32_t dlo, dhi;              // data index bytes (>= 0x80: null / pilot), j = 0..3 and 4..7
    uint32_t lneg, lnul;            // bit j: L < 0, L == 0
};
__device__ __forceinline__ SweepLane make_sweep_lane(int u)
{
    SweepLane c = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const uint32_t d = (uint32_t)(uint8_t)c_tab.bin_data[u + 8 * j];
        if (j < 4) c.dlo |= d << (8 * j); else c.dhi |= d << (8 * (j - 4));
        const int l = c_tab.bin_lts[u + 8 * j];
        c.lneg |= (uint32_t)(l < 0) << j; c.lnul |= (uint32_t)(l == 0) << j;
    }
    return c;
}
struct SweepFrame {                 // one frame's inputs
    const float2 *x; const float *g; const uint32_t *bits;
    int n_sym; double sigma_d; uint32_t seed, stream; uint64_t frame_id;
    unsigned long long *replayed;
};
struct SweepTotals { uint32_t i, q, both; float e2; };

// One frame in the reference's arithmetic, samples straight from global memory (the replay of k_stream_rxn<kArithChecked>).
template <int NOISE>
__device__ __noinline__ SweepTotals sweep_frame_replay(SweepFrame fr, float2 *tile_w, float2 *lts /* [2][kWin] */)
{
    const int lane = threadIdx.x & 31, grp = lane >> 3, u = lane & 7;
    float2 *tile = tile_w + grp * kGroupPitch;
    Tw<true> tw; tw.load(u);
    const SweepLane sl = make_sweep_lane(u);
    const int n_sym = fr.n_sym;
    const int n_pass = 1 + (n_sym > 2 ? (n_sym + 1) / 4 : 0);
    SweepTotals t = {0u, 0u, 0u, 0.f};
    unsigned long long *replayed = fr.replayed;
    for (int pass = 0; pass < n_pass; ++pass) {
        const int sym = pass == 0 ? grp - 2 : 2 + (pass - 1) * 4 + grp;     // < 0: LTS half
        const bool active = sym < n_sym;
        const int n0 = sym < 0 ? 32 + 64 * grp : 176 + 80 * sym;           // Channel_Estimation :837-838, CP strip :1028
        float z[8];
        if (NOISE == kNoisePhilox && active) {
            const int base = window_block_base(n0) + u;
            float za[4], zb[4];
            philox_normals4(fr.seed, fr.stream, fr.frame_id, (uint32_t)base, kDomainNoise, za);
            philox_normals4(fr.seed, fr.stream, fr.frame_id, (uint32_t)(base + 8), kDomainNoise, zb);
#pragma unroll
            for (int m = 0; m < 4; ++m) { z[m] = za[m]; z[4 + m] = zb[m]; }
        }
        float2 v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int m = slot_m<true>(i);
            float2 sm = make_float2(0.f, 0.f);
            if (active) {
                sm = fr.x[n0 + u + 8 * m];
                if (NOISE == kNoiseInject) sm.x = add_noise<true>(sm.x, fr.g[n0 + u + 8 * m], fr.sigma_d, 0.f);
                if (NOISE == kNoisePhilox) sm.x = add_noise<true>(sm.x, z[m], fr.sigma_d, 0.f);
            }
            v[i] = sm;
        }
        fft64<true>(v, tw, tile, u);
        if (pass == 0 && grp < 2) {
#pragma unroll
            for (int j = 0; j < 8; ++j) lts[grp * kWin + u + 8 * j] = v[j];
        }
        __syncwarp();
        if (sym >= 0 && active) {
            const uint32_t *w = fr.bits + sym * 3;
            const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
            uint32_t pk = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const uint32_t d = ((j < 4 ? sl.dlo : sl.dhi) >> (8 * (j & 3))) & 0xFFu;
                const float sc = ((sl.lnul >> j) & 1u) ? 0.f : (((sl.lneg >> j) & 1u) ? -0.5f : 0.5f);
                const float2 A = lts[u + 8 * j], B = lts[kWin + u + 8 * j];
                const float2 Hh = make_float2(__fmul_rn(__fadd_rn(A.x, B.x), sc), __fmul_rn(__fadd_rn(A.y, B.y), sc));      // :848
                pk += process_bin_hot<true>(v[j], Hh, sc, bit_pair(w0, w1, w2, (int)d), d < 0x80u, t.e2);
            }
            t.i += pk & 0xFFu; t.q += (pk >> 8) & 0xFFu; t.both += pk >> 16;
        }
        __syncwarp();
    }
    if (lane == 0 && replayed != nullptr) atomicAdd(replayed, 1ull);
    return t;
}

template <int ARITH, int NOISE>
__global__ void __launch_bounds__(kThreads, 2) k_stream_rxn(RxParams p)
{
    constexpr bool EXACT = ARITH == kArithExact, CHECKED = ARITH == kArithChecked;
    constexpr bool SPEC = ARITH != kArithExact;                 // see k_stream_rx2
    constexpr int LEVEL = CHECKED ? 2 : 1;
    extern __shared__ __align__(128) unsigned char s_raw[];
    __shared__ unsigned long long s_cnt[kWarpsPerBlock][4];
    __shared__ double s_sum[kWarpsPerBlock][2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, u = lane & 7;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);                  // same value, provably warp-uniform
    using SW = StreamWarp<NOISE == kNoiseInject>;
    using SS = StreamStage<NOISE == kNoiseInject>;
    SW &ws = reinterpret_cast<SW *>(s_raw)[warp];
    SW &ws_u = reinterpret_cast<SW *>(s_raw)[warp_u];
    float2 *tile = ws.tile + grp * kGroupPitch;
    Tw<EXACT> tw; tw.load(u);
    const ItemConst ic = make_items(lane);
    const int n_sym = p.n_sym, len = 160 + 80 * n_sym;
    const int n_pass = 1 + (n_sym > 2 ? (n_sym + 1) / 4 : 0);
    const long stride = (long)gridDim.x * kWarpsPerBlock;
    const long f_first = (long)blockIdx.x * kWarpsPerBlock + warp_u;
    const int my_frames = f_first < p.n_frames ? (int)((p.n_frames - f_first + stride - 1) / stride) : 0;   // < 2^31 by a wide margin
    const double q = (double)kQpsk;
    const double ref2_frame = 48.0 * n_sym * (2.0 * q * q);
    const float inv_ref2 = (float)(1.0 / ref2_frame);

    const uint32_t stage0 = tma::saddr(&ws_u.st[0]);
    const uint32_t bar0 = tma::saddr(&ws_u.bar[0]);
    // refill stage s with pass `pass` of this warp's frame number jf: only the windows that exist are fetched
    auto issue = [&](int jf, int pass, int s) {
        if (tma::elect_one()) {
            const long f = f_first + (long)jf * stride;
            const int first_sym = pass == 0 ? 0 : 2 + 4 * (pass - 1);
            const int left = n_sym - first_sym;
            const int nwin = pass == 0 ? 2 + (left < 2 ? left : 2) : (left < 4 ? left : 4);
            const int n0 = pass == 0 ? 32 : 176 + 80 * first_sym, n1 = pass == 0 ? 96 : n0 + 80;
            const int n2 = pass == 0 ? 176 : n0 + 160, n3 = n2 + 80;
            const uint32_t bar = bar0 + 8u * (uint32_t)s;
            const uint32_t dst = stage0 + (uint32_t)s * (uint32_t)sizeof(SS);
            const char *x = reinterpret_cast<const char *>(p.in) + f * ((long)len * 8);
            tma::expect_tx_addr(bar, (uint32_t)nwin * (NOISE == kNoiseInject ? 768u : 512u));
            tma::bulk_addr(dst + 0 * kWin * 8, x + n0 * 8, 512, bar);
            if (nwin > 1) tma::bulk_addr(dst + 1 * kWin * 8, x + n1 * 8, 512, bar);
            if (nwin > 2) tma::bulk_addr(dst + 2 * kWin * 8, x + n2 * 8, 512, bar);
            if (nwin > 3) tma::bulk_addr(dst + 3 * kWin * 8, x + n3 * 8, 512, bar);
            if (NOISE == kNoiseInject) {
                const char *g = reinterpret_cast<const char *>(p.g) + f * ((long)len * 4);
                const uint32_t gd = dst + 4 * kWin * 8;
                tma::bulk_addr(gd + 0 * kWin * 4, g + n0 * 4, 256, bar);
                if (nwin > 1) tma::bulk_addr(gd + 1 * kWin * 4, g + n1 * 4, 256, bar);
                if (nwin > 2) tma::bulk_addr(gd + 2 * kWin * 4, g + n2 * 4, 256, bar);
                if (nwin > 3) tma::bulk_addr(gd + 3 * kWin * 4, g + n3 * 4, 256, bar);
            }
        }
    };
    if (lane == 0) {
        for (int s = 0; s < kStages; ++s) tma::mbar_init(&ws.bar[s], 1);
        tma::fence_mbar_init();
    }
    __syncwarp();
    // the unit to refill next: (frame number, pass)
    int jf_issue = 0, pass_issue = 0;
    auto issue_next = [&](int s) {
        if (jf_issue < my_frames) {
            issue(jf_issue, pass_issue, s);
            if (++pass_issue == n_pass) { pass_issue = 0; ++jf_issue; }
        }
    };
    for (int s = 0; s < kStages; ++s) issue_next(s);

    uint32_t a_i = 0, a_q = 0, a_both = 0, a_ferr = 0, a_frames = 0;
    double a_e2 = 0.0, a_evm = 0.0;
    uint32_t k = 0;                                        // units consumed (ring position)
    for (int j_chunk = 0; j_chunk < my_frames; j_chunk += 32) {
        double sig_mine = 0.0;
        if (NOISE != kNoiseNone) {
            const int jl = j_chunk + lane;
            if (jl < my_frames) sig_mine = __dsqrt_rn((double)__fdiv_rn(p.power[f_first + (long)jl * stride], p.snr_lin));   // :647, :651
        }
        float c_e2 = 0.f, c_evm = 0.f;
        for (int kk = 0; kk < 32; ++kk) {
            const int jf = j_chunk + kk;
            if (jf >= my_frames) break;
            const long f = f_first + (long)jf * stride;
            const double sigma_d = NOISE != kNoiseNone ? __shfl_sync(0xffffffffu, sig_mine, kk) : 0.0;
            const float sigma_f = (float)sigma_d;
            const uint32_t *fbits = p.tx_bits + f * ((long)n_sym * 3);
            uint32_t f_i = 0, f_q = 0, f_both = 0;
            float f_e2 = 0.f, rH2 = 0.f;
            bool doubt = false;
            for (int pass = 0; pass < n_pass; ++pass, ++k) {
                const int s = (int)(k & 1u);
                const uint32_t phase = (k >> 1) & 1u;
                const int sym = pass == 0 ? grp - 2 : 2 + (pass - 1) * 4 + grp;     // < 0: LTS half
                const bool active = sym < n_sym;
                float z[8];
                if (NOISE == kNoisePhilox && active) {
                    const int blk = window_block_base(sym < 0 ? 32 + 64 * grp : 176 + 80 * sym) + u;
                    float za[4], zb[4];
                    philox_normals4(p.seed, p.stream, p.frame0 + (uint64_t)f, (uint32_t)blk, kDomainNoise, za);
                    philox_normals4(p.seed, p.stream, p.frame0 + (uint64_t)f, (uint32_t)(blk + 8), kDomainNoise, zb);
#pragma unroll
                    for (int m = 0; m < 4; ++m) { z[m] = za[m]; z[4 + m] = zb[m]; }
                }
                // this pass's payload words for the lane's items (used after the transform): round 0 and, from pass 1 on, round 1
                const int first_sym = pass == 0 ? 0 : 2 + (pass - 1) * 4;
                const uint32_t *fb = fbits + first_sym * 3;
                const int left = pass == 0 ? (n_sym < 2 ? n_sym : 2) : n_sym - first_sym;     // symbols this pass decides
                uint32_t wq[6], vmask = 0;                                                   // bit t: item t of this pass exists
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const int s01 = ic.f_off[t] < kWin ? 0 : 1;
                    const bool v0 = s01 < left, v1 = 2 + s01 < left;
                    wq[t] = v0 ? fb[ic.word[t]] : 0u;
                    wq[3 + t] = v1 ? fb[6 + ic.word[t]] : 0u;
                    vmask |= (uint32_t)v0 << t | (uint32_t)v1 << (3 + t);
                }
                tma::wait_addr(bar0 + 8u * (uint32_t)s, phase);
                float2 v[8];
                float2 n2 = make_float2(0.f, 0.f);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int m = slot_m<EXACT>(i);
                    float2 smp = make_float2(0.f, 0.f);
                    if (active) {
                        smp = ws.st[s].x[grp][u + 8 * m];
                        if (NOISE == kNoiseInject) smp.x = add_noise<EXACT>(smp.x, ws.st[s].g[grp][u + 8 * m], sigma_d, sigma_f);   // CHECKED: speculated
                        if (NOISE == kNoisePhilox) smp.x = add_noise<EXACT>(smp.x, z[m], sigma_d, sigma_f);
                    }
                    if (SPEC) n2 = __ffma2_rn(smp, smp, n2);
                    v[i] = smp;
                }
                __syncwarp();                                     // every lane has its samples: the stage can be refilled
                issue_next(s);
                fft64<EXACT>(v, tw, tile, u);
                float rad = 0.f;
                if (SPEC) rad = window_radius(n2, p.radius_scale, NOISE != kNoiseNone ? p.radius_chan * sigma_f : 0.f);
                uint32_t pk = 0;
                if (pass == 0) {
                    float2 *dst = grp < 2 ? ws.lts[grp] : ws.tile + (grp - 2) * kWin;
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) dst[u + 8 * jj] = v[jj];
                    if (SPEC && u == 0) ws.radius[grp] = rad;
                    __syncwarp();
                    float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (SPEC) {
                        r4 = *reinterpret_cast<const float4 *>(ws.radius);
                        rH2 = r4.x + r4.y;                                        // 2 r_H, kept for the frame's later passes
                    }
                    const float den_min4 = (p.evm_guard * rH2) * (p.evm_guard * rH2);
#pragma unroll
                    for (int t = 0; t < 3; ++t) {
                        const int isym = ic.f_off[t] < kWin ? 0 : 1;              // the item's symbol
                        const bool valid = (vmask >> t) & 1u;
                        const float2 A = ws.lts[0][ic.bin[t]], B = ws.lts[1][ic.bin[t]];
                        const uint32_t w = wq[t];
                        float e2 = 0.f;
                        uint32_t r;
                        if (SPEC) {
                            bool dbt = false;
                            float2 e2v = make_float2(0.f, 0.f);
                            r = process_bin_spec<LEVEL>(ws.tile[ic.f_off[t]], cadd(A, B), 4.f * ic.sc[t], w >> ic.shift[t],
                                                    isym == 0 ? r4.z : r4.w, rH2, den_min4, e2v, dbt);
                            e2 = e2v.x + e2v.y;
                            doubt = doubt || (valid && dbt);
                        } else {
                            const float2 Hh = make_float2(__fmul_rn(__fadd_rn(A.x, B.x), ic.sc[t]), __fmul_rn(__fadd_rn(A.y, B.y), ic.sc[t]));   // :848
                            r = item_eval<EXACT>(ws.tile[ic.f_off[t]], Hh, ic.sc[t], w >> ic.shift[t], e2);
                        }
                        pk += valid ? r : 0u; f_e2 += valid ? e2 : 0.f;
                    }
                } else {
                    // four symbols: all groups publish F, then the 192 data bins are dealt out in two rounds of three items per
                    // lane -- the item pattern of round 1 is that of round 0 two symbols (= two windows, six payload words) up
                    float2 *dst = ws.tile + grp * kWin;
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) dst[u + 8 * jj] = v[jj];
                    if (SPEC && u == 0) ws.radius[grp] = rad;
                    __syncwarp();
                    float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (SPEC) r4 = *reinterpret_cast<const float4 *>(ws.radius);
                    const float den_min4 = (p.evm_guard * rH2) * (p.evm_guard * rH2);
#pragma unroll
                    for (int round = 0; round < 2; ++round) {
#pragma unroll
                        for (int t = 0; t < 3; ++t) {
                            const int isym = ic.f_off[t] < kWin ? 0 : 1;
                            const bool valid = (vmask >> (3 * round + t)) & 1u;
                            const float2 A = ws.lts[0][ic.bin[t]], B = ws.lts[1][ic.bin[t]];
                            const uint32_t w = wq[3 * round + t];
                            const float2 F = ws.tile[2 * round * kWin + ic.f_off[t]];
                            float e2 = 0.f;
                            uint32_t r;
                            if (SPEC) {
                                bool dbt = false;
                                float2 e2v = make_float2(0.f, 0.f);
                                const float rF = round == 0 ? (isym == 0 ? r4.x : r4.y) : (isym == 0 ? r4.z : r4.w);
                                r = process_bin_spec<LEVEL>(F, cadd(A, B), 4.f * ic.sc[t], w >> ic.shift[t], rF, rH2, den_min4, e2v, dbt);
                                e2 = e2v.x + e2v.y;
                                doubt = doubt || (valid && dbt);
                            } else {
                                const float2 Hh = make_float2(__fmul_rn(__fadd_rn(A.x, B.x), ic.sc[t]), __fmul_rn(__fadd_rn(A.y, B.y), ic.sc[t]));   // :848
                                r = item_eval<EXACT>(F, Hh, ic.sc[t], w >> ic.shift[t], e2);
                            }
                            pk += valid ? r : 0u; f_e2 += valid ? e2 : 0.f;
                        }
                    }
                }
                f_i += pk & 0xFFu; f_q += (pk >> 8) & 0xFFu; f_both += pk >> 16;
                __syncwarp();
            }
            if (SPEC) {
                if (__any_sync(0xffffffffu, doubt)) {             // not provably the reference's decisions: replay the frame exactly
                    SweepFrame fr;
                    fr.x = p.in + f * len; fr.g = NOISE == kNoiseInject ? p.g + f * len : nullptr; fr.bits = fbits; fr.n_sym = n_sym;
                    fr.sigma_d = sigma_d; fr.seed = p.seed; fr.stream = p.stream; fr.frame_id = p.frame0 + (uint64_t)f; fr.replayed = p.replayed;
                    const SweepTotals t = sweep_frame_replay<NOISE>(fr, ws.tile, &ws.lts[0][0]);
                    f_i = t.i; f_q = t.q; f_both = t.both; f_e2 = t.e2;
                }
            }
            const bool any_err = __any_sync(0xffffffffu, (f_i | f_q) != 0u);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) f_e2 += __shfl_xor_sync(0xffffffffu, f_e2, o);
            float evm;
            asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(evm) : "f"(f_e2 * inv_ref2));                                              // :1124
            a_i += f_i; a_q += f_q; a_both += f_both;
            a_ferr += any_err; a_frames += 1;
            c_e2 += f_e2; c_evm += evm;
        }
        a_e2 += (double)c_e2; a_evm += (double)c_evm;
    }
    if (p.counters == nullptr) return;
    const uint32_t t_i = warp_sum(a_i), t_q = warp_sum(a_q), t_both = warp_sum(a_both);
    if (lane == 0) {
        s_cnt[warp][0] = (unsigned long long)t_i + 2ull * t_q - 2ull * t_both;     // bit errors (map of :423-430)
        s_cnt[warp][1] = (unsigned long long)t_i + t_q;
        s_cnt[warp][2] = a_ferr; s_cnt[warp][3] = a_frames;
        s_sum[warp][0] = a_e2; s_sum[warp][1] = a_evm;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long c[4] = {0, 0, 0, 0}; double sm[2] = {0, 0};
        for (int w = 0; w < kWarpsPerBlock; ++w) {
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

template <int NOISE> inline size_t stream_smem_bytes() { return sizeof(StreamWarp<NOISE == kNoiseInject>) * kWarpsPerBlock; }

}  // namespace ofdm

namespace ofdm {
// ------------------------------------------------------------------------------------------------
// configs[4] extension (no counterpart in the reference, SURVEY Q8): per-frame multipath channel
// y[n] = sum_l h[l] x[n-l], x[n<0] = 0, n_taps <= 16 = CP length (no inter-symbol interference, the LTS
// estimate + one-tap equaliser of :830-850, :1046-1052 absorb it).  Taps are either supplied
// ([frames][n_taps] complex) or drawn on chip: i.i.d. complex Gaussian, E|h_l|^2 = 1/n_taps, Philox domain 2,
// tap l = normals (2l, 2l+1) of block l/2.  Same float operation order as the oracle (orc_apply_taps):
// descending l, separate multiplies and adds (no FMA), so supplied taps reproduce it bit for bit.

// The FIR-type kernels below (multipath taps, RRC shaping, matched filter) stage a frame through shared memory in tiles of
// `tile` samples plus the filter's halo, one tile per warp and pass, so that the shared-memory footprint does not grow with the
// frame length (any n_sym up to OFDM_MAX_SYM, any capture length); every output sample is still accumulated by one thread in
// the reference's order, so tiling does not change a bit.
constexpr int kFirTile = 2048;          // largest tile (samples per warp and pass)
constexpr int kFirHalo = 32;            // room for the halo: 15 taps back (multipath), 20 samples back (RRC)
inline int fir_tile(int samples) { int t = (samples + 31) & ~31; return t < kFirTile ? t : kFirTile; }
inline size_t fir_smem_bytes(int tile) { return (size_t)kWarpsPerBlock * (tile + kFirHalo) * sizeof(float2); }

template <bool PHILOX>
__global__ void __launch_bounds__(kThreads) k_multipath(const float2 *__restrict__ tx, const float2 *__restrict__ taps, uint32_t seed,
                                                        uint64_t frame0, int n_taps, float2 *__restrict__ out, float2 *__restrict__ taps_out,
                                                        long n_frames, int len, int tile)
{
    extern __shared__ __align__(128) unsigned char s_raw[];
    __shared__ float2 s_taps[kWarpsPerBlock][kMaxTaps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float2 *sx = reinterpret_cast<float2 *>(s_raw) + (size_t)warp * (tile + kFirHalo);
    float2 *sh = s_taps[warp];
    const float scale = sqrtf(0.5f / (float)n_taps);
    for (long f = (long)blockIdx.x * kWarpsPerBlock + warp; f < n_frames; f += (long)gridDim.x * kWarpsPerBlock) {
        const float2 *x = tx + f * len;
        if (PHILOX) {
            if (2 * lane < n_taps) {
                float z[4];
                philox_normals4(seed, 0u, frame0 + (uint64_t)f, (uint32_t)lane, kDomainTaps, z);
                sh[2 * lane] = make_float2(scale * z[0], scale * z[1]);
                if (2 * lane + 1 < n_taps) sh[2 * lane + 1] = make_float2(scale * z[2], scale * z[3]);
            }
        } else if (lane < n_taps) sh[lane] = taps[f * n_taps + lane];
        __syncwarp();
        if (taps_out != nullptr && lane < n_taps) taps_out[f * n_taps + lane] = sh[lane];
        for (int n0 = 0; n0 < len; n0 += tile) {
            const int n1 = n0 + tile < len ? n0 + tile : len;
            const int lo = n0 - (kMaxTaps - 1) > 0 ? n0 - (kMaxTaps - 1) : 0;        // halo: the taps reach 15 samples back
            for (int i = lo + lane; i < n1; i += 32) sx[i - lo] = x[i];
            __syncwarp();
            for (int n = n0 + lane; n < n1; n += 32) {
                float ar = 0.f, ai = 0.f;
                for (int l = (n_taps - 1 < n ? n_taps - 1 : n); l >= 0; --l) {
                    const float2 a = sx[n - l - lo], b = sh[l];
                    ar = __fadd_rn(ar, __fsub_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)));
                    ai = __fadd_rn(ai, __fadd_rn(__fmul_rn(a.x, b.y), __fmul_rn(a.y, b.x)));
                }
                out[f * len + n] = make_float2(ar, ai);
            }
            __syncwarp();
        }
    }
}

// ofdm_counters is 5 x u64 + 3 x double per SNR point; collectives want homogeneous buffers
__global__ void k_counters_pack(const ofdm_counters *__restrict__ c, int n, unsigned long long *__restrict__ ints, double *__restrict__ dbls)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const ofdm_counters v = c[i];
    ints[5 * i] = v.bit_errors; ints[5 * i + 1] = v.bits; ints[5 * i + 2] = v.frames_in_error; ints[5 * i + 3] = v.rail_errors; ints[5 * i + 4] = v.frames;
    dbls[3 * i] = v.sum_err2; dbls[3 * i + 1] = v.sum_ref2; dbls[3 * i + 2] = v.sum_evm_lin;
}
__global__ void k_counters_unpack(ofdm_counters *__restrict__ c, int n, const unsigned long long *__restrict__ ints, const double *__restrict__ dbls)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ofdm_counters v;
    v.bit_errors = ints[5 * i]; v.bits = ints[5 * i + 1]; v.frames_in_error = ints[5 * i + 2]; v.rail_errors = ints[5 * i + 3]; v.frames = ints[5 * i + 4];
    v.sum_err2 = dbls[3 * i]; v.sum_ref2 = dbls[3 * i + 1]; v.sum_evm_lin = dbls[3 * i + 2];
    c[i] = v;
}

// ------------------------------------------------------------------------------------------------
// SURVEY 8(f) rank 1: pulse shaping.  x2 zero-stuff + 21-tap RRC on the way out (OFDM.c:587-605), matched filter +
// decimation on the way in (OFDM.c:959-996), both as the reference's Convolution() (:342-364) accumulates them:
// float, input index ascending, real taps (RRC_Filter_Tx :32) so each product is (a*h, b*h).  Zero-stuffed inputs
// contribute exact zeros and are skipped.  One warp per frame, frame staged in shared memory, coalesced stores.
__constant__ float c_rrc[21] = {-0.000454720514876223f, 0.00353689555574986f, -0.00714560809091226f, 0.00757906190517828f,
                                0.00214368242727367f, -0.0106106866672496f, 0.0300115539818315f, -0.0530534333362480f,
                                -0.0750288849545787f, 0.409168714634052f, 0.803738600397980f, 0.409168714634052f,
                                -0.0750288849545787f, -0.0530534333362480f, 0.0300115539818315f, -0.0106106866672496f,
                                0.00214368242727367f, 0.00757906190517828f, -0.00714560809091226f, 0.00353689555574986f,
                                -0.000454720514876223f};

__global__ void __launch_bounds__(kThreads) k_rrc_tx(const float2 *__restrict__ frames, float2 *__restrict__ out, long n_frames, int len, int tile)
{
    extern __shared__ __align__(128) unsigned char s_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float2 *sx = reinterpret_cast<float2 *>(s_raw) + (size_t)warp * (tile + kFirHalo);
    const int n_out = 2 * len + 20;
    for (long f = (long)blockIdx.x * kWarpsPerBlock + warp; f < n_frames; f += (long)gridDim.x * kWarpsPerBlock) {
        for (int k0 = 0; k0 < n_out; k0 += 2 * tile) {                        // 2 * tile outputs need tile + 10 inputs
            const int k1 = k0 + 2 * tile < n_out ? k0 + 2 * tile : n_out;
            const int j_lo = k0 >= 20 ? (k0 - 19) / 2 : 0;                    // first input sample (index i / 2) any of these outputs reads
            const int j_hi = (k1 - 1) / 2 < len - 1 ? (k1 - 1) / 2 : len - 1;
            for (int j = j_lo + lane; j <= j_hi; j += 32) sx[j - j_lo] = frames[f * len + j];
            __syncwarp();
            for (int k = k0 + lane; k < k1; k += 32) {
                const int lo = k - 20 < 0 ? 0 : k - 20, hi = k < 2 * len - 1 ? k : 2 * len - 1;
                float ar = 0.f, ai = 0.f;
                for (int i = lo + (lo & 1); i <= hi; i += 2) {                // even (non-stuffed) inputs, ascending
                    const float2 a = sx[(i >> 1) - j_lo];
                    const float h = c_rrc[k - i];
                    ar = __fadd_rn(ar, __fmul_rn(a.x, h)); ai = __fadd_rn(ai, __fmul_rn(a.y, h));
                }
                out[f * n_out + k] = make_float2(ar, ai);
            }
            __syncwarp();
        }
    }
}

// matched filter + decimation (:965, :986-996): output r reads the filtered sample k = p0 + 2 r, i.e. inputs k - 20 .. k.
// idx == nullptr: the same packet index for every capture (ofdm_rrc_rx); else per capture (:978), and filtered samples
// past the end of the capture (which the reference would read out of bounds when a packet starts late) count as zero.
__global__ void __launch_bounds__(kThreads) k_rrc_rx(const float2 *__restrict__ in, const int32_t *__restrict__ idx, int packet_idx,
                                                     float2 *__restrict__ out, long n_frames, int in_len, int frame_len, int tile)
{
    extern __shared__ __align__(128) unsigned char s_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float2 *sx = reinterpret_cast<float2 *>(s_raw) + (size_t)warp * (tile + kFirHalo);
    const int r_tile = tile / 2;                                              // tile / 2 outputs need tile + 20 inputs
    for (long f = (long)blockIdx.x * kWarpsPerBlock + warp; f < n_frames; f += (long)gridDim.x * kWarpsPerBlock) {
        const int p0 = idx != nullptr ? idx[f] : packet_idx;
        for (int r0 = 0; r0 < frame_len; r0 += r_tile) {
            const int r1 = r0 + r_tile < frame_len ? r0 + r_tile : frame_len;
            const int i_lo = p0 + 2 * r0 - 20 > 0 ? p0 + 2 * r0 - 20 : 0;
            const int i_hi = p0 + 2 * (r1 - 1) < in_len - 1 ? p0 + 2 * (r1 - 1) : in_len - 1;
            for (int i = i_lo + lane; i <= i_hi; i += 32) sx[i - i_lo] = in[f * in_len + i];
            __syncwarp();
            for (int r = r0 + lane; r < r1; r += 32) {
                const int k = p0 + 2 * r;                                     // :992-996
                float ar = 0.f, ai = 0.f;
                if (k < in_len + 20) {
                    const int lo = k - 20 < 0 ? 0 : k - 20, hi = k < in_len - 1 ? k : in_len - 1;
                    for (int i = lo; i <= hi; ++i) {
                        const float2 a = sx[i - i_lo];
                        const float h = c_rrc[k - i];
                        ar = __fadd_rn(ar, __fmul_rn(a.x, h)); ai = __fadd_rn(ai, __fmul_rn(a.y, h));
                    }
                }
                out[f * frame_len + r] = make_float2(ar, ai);
            }
            __syncwarp();
        }
    }
}

// ------------------------------------------------------------------------------------------------
// SURVEY 8(f) rank 2: packet detection and selection (OFDM.c:659-771), batched over captures.
// Detection: delay 16, window 32, NO conjugate (as the reference and its MATLAB model).  Per lag i the reference
// accumulates 32 float complex products sequentially and a float "peak" fed with double cabs()^2 terms, then
// out_i = (float)(cabs(corr)^2 / (double)(float)(peak*peak)); the sequential float sums differ per lag, so there is
// no sliding-window reuse of the sums if the bits are to match.  What the lags do share is the summands: the float
// product rx[n] * rx[n+16] (separately rounded multiplies, :674) and the double term cabs(rx[n])^2 (glibc hypot, :675) are
// computed once per sample and staged in shared memory; each thread then runs its lag's two 32-term chains over them.
// A capture is worked through in tiles of `tile` lags (+ 47 samples of halo), so that the footprint does not depend on its length.
__global__ void __launch_bounds__(kThreads) k_packet_detect(const float2 *__restrict__ rx, float *__restrict__ corr, long n, int len, int tile)
{
    extern __shared__ __align__(128) unsigned char s_raw[];
    double *pk2 = reinterpret_cast<double *>(s_raw);
    float2 *prod = reinterpret_cast<float2 *>(pk2 + tile + 48);
    const int n_corr = len - 47;
    for (long c = blockIdx.x; c < n; c += gridDim.x) {
        const float2 *x = rx + c * len;
        for (int i0 = 0; i0 < n_corr; i0 += tile) {
            const int i1 = i0 + tile < n_corr ? i0 + tile : n_corr;
            for (int sidx = i0 + threadIdx.x; sidx < i1 + 47; sidx += kThreads) {        // samples i0 .. i1 + 46 (< len)
                const float2 a = x[sidx];
                const double h = hypot_glibc((double)a.x, (double)a.y);          // cabs :675
                pk2[sidx - i0] = __dmul_rn(h, h);
                if (sidx + 16 < len) {
                    const float2 b = x[sidx + 16];
                    prod[sidx - i0] = make_float2(__fsub_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)),      // :674, float complex multiply
                                                  __fadd_rn(__fmul_rn(a.x, b.y), __fmul_rn(a.y, b.x)));
                }
            }
            __syncthreads();
            for (int i = i0 + threadIdx.x; i < i1; i += kThreads) {
                float cr = 0.f, ci = 0.f, peak = 0.f;
#pragma unroll 8
                for (int k = 0; k < 32; ++k) {
                    const float2 t = prod[i - i0 + k];
                    cr = __fadd_rn(cr, t.x);
                    ci = __fadd_rn(ci, t.y);
                    peak = __double2float_rn(__dadd_rn((double)peak, pk2[i - i0 + k + 16]));           // :675
                }
                const double hc = hypot_glibc((double)cr, (double)ci);
                corr[c * n_corr + i] = __double2float_rn(__ddiv_rn(__dmul_rn(hc, hc), (double)__fmul_rn(peak, peak)));   // :677
            }
            __syncthreads();
        }
    }
}

// Selection OFDM.c:685-771: indices above 0.75; a gap > 300 to the previous one opens a candidate; all candidates but
// the last are tried in order and the first whose correlation 230 lags later is still above the threshold wins:
// packet_idx = candidate + len_RRC_rx + 1 (= +11); 0 if none.  One thread per capture (the scan is sequential).
__global__ void __launch_bounds__(kThreads) k_packet_select(const float *__restrict__ corr, int32_t *__restrict__ idx_out, long n, int len_corr)
{
    // One warp per capture, 32 lags per step (coalesced); everything below the ballot is warp-uniform.  Within a step only
    // the first lag above the threshold can open a candidate (the others follow within 32 < 300 lags).  A candidate is tried
    // when the next one appears, so the last one never is -- "x < packet_front_count - 1" (:754).
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (long c = (long)blockIdx.x * kWarpsPerBlock + warp; c < n; c += (long)gridDim.x * kWarpsPerBlock) {
        const float *x = corr + c * len_corr;
        int prev = -1, pending = -1, result = 0;
        for (int base = 0; base < len_corr && result == 0; base += 32) {
            const int i = base + lane;
            const bool above = i < len_corr && fabsf(x[i]) > 0.75f;
            const uint32_t mask = __ballot_sync(0xffffffffu, above);
            if (mask == 0u) continue;
            const int first = base + __ffs((int)mask) - 1;
            if (first - prev > 300) {                                            // a new candidate: the pending one is not the last
                if (pending >= 0) {
                    const int look = pending + 230;                              // :756 (unchecked in the reference)
                    if (look < len_corr && fabsf(x[look]) > 0.75f) result = pending + 11;     // :758
                }
                pending = first;
            }
            prev = base + 31 - __clz((int)mask);
        }
        if (lane == 0) idx_out[c] = result;
    }
}

// ------------------------------------------------------------------------------------------------
// SURVEY 8(f) ranks 3 and 4: CFO estimation / correction (OFDM.c:773-828) and the glue of the reference's full
// over-the-air path (STS slot :483-492/:572, 10x repetition :607-612, capture window :945-955, per-packet
// decimation :986-996).
//
// CFO: the correlation sum_i a[i]*conj(b[i]) uses the DOUBLE conj(), so every product is formed in double and the
// float complex accumulator takes (float)((double)acc + product), sequentially (lane 0).  freq = (float)(K * atan2)
// and the rotator cexp(-I*2*PI*f*ts*i) are double libm calls in the reference: the device's atan2 / sincos agree
// with glibc to an ulp of double, which the following roundings to float absorb except with probability ~1e-8 per
// sample -- this stage is specified to 1e-6 relative, not bit-exact.  Coarse: slots 5/6 of the STS (samples 80..111),
// product with the rotator in double.  Fine: the LTS halves (192..319), rotator rounded to float first (exp_term),
// product in float.
template <bool FINE>
__global__ void __launch_bounds__(kThreads) k_cfo(const float2 *__restrict__ rx, float2 *__restrict__ out, float *__restrict__ freq_out,
                                                  long n, int len)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int kA = FINE ? 192 : 80, kB = FINE ? 256 : 96, kN = FINE ? 64 : 16;
    constexpr double kPi = 3.14159265358979323846, kTs = 1 / 20e6;                       // PI :13, ts_sec :17
    const double kScale = -1.0 / (2 * kPi * kN * kTs);                                   // :798 / :821
    for (long f = (long)blockIdx.x * kWarpsPerBlock + warp; f < n; f += (long)gridDim.x * kWarpsPerBlock) {
        const float2 *x = rx + f * len;
        float fr = 0.f;
        if (lane == 0) {
            float accr = 0.f, acci = 0.f;
            for (int i = 0; i < kN; ++i) {
                const float2 a = x[kA + i], b = x[kB + i];
                const double ar = a.x, ai = a.y, br = b.x, nbi = -(double)b.y;
                const double pr = __dsub_rn(__dmul_rn(ar, br), __dmul_rn(ai, nbi)), pi = __dadd_rn(__dmul_rn(ar, nbi), __dmul_rn(ai, br));
                accr = __double2float_rn(__dadd_rn((double)accr, pr));
                acci = __double2float_rn(__dadd_rn((double)acci, pi));
            }
            fr = __double2float_rn(__dmul_rn(kScale, atan2((double)acci, (double)accr)));
            if (freq_out != nullptr) freq_out[f] = fr;
        }
        fr = __shfl_sync(0xffffffffu, fr, 0);
        const double w = __dmul_rn(__dmul_rn(__dmul_rn(-2.0, kPi), (double)fr), kTs);   // ((-2*PI)*f)*ts, the reference's association
        for (int i = lane; i < len; i += 32) {
            double s, c;
            sincos(__dmul_rn(w, (double)i), &s, &c);
            const float2 v = x[i];
            float2 y;
            if (FINE) {
                const float cf = __double2float_rn(c), sf = __double2float_rn(s);
                y.x = __fsub_rn(__fmul_rn(v.x, cf), __fmul_rn(v.y, sf));
                y.y = __fadd_rn(__fmul_rn(v.x, sf), __fmul_rn(v.y, cf));
            } else {
                y.x = __double2float_rn(__dsub_rn(__dmul_rn((double)v.x, c), __dmul_rn((double)v.y, s)));
                y.y = __double2float_rn(__dadd_rn(__dmul_rn((double)v.x, s), __dmul_rn((double)v.y, c)));
            }
            out[f * len + i] = y;
        }
    }
}

// out[f][j] = in[f][(start_f + j) % in_len], j < out_len: Slice_Repeater (:193) generalised -- prefix slices (:955),
// tiling (:612: start 0, out_len = r * in_len) and capture windows of the repeated waveform all come out of it.
// One warp per frame: 32-bit index arithmetic, the wrap kept incrementally (no division per sample).
__global__ void __launch_bounds__(kThreads) k_gather(const float2 *__restrict__ in, const int32_t *__restrict__ start, int start_scalar,
                                                     float2 *__restrict__ out, long n, int in_len, int out_len)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int step = 32 % in_len;
    for (long f = (long)blockIdx.x * kWarpsPerBlock + warp; f < n; f += (long)gridDim.x * kWarpsPerBlock) {
        const int s = start != nullptr ? start[f] : start_scalar;
        const float2 *src = in + f * in_len;
        float2 *dst = out + f * out_len;
        int idx = (int)(((long)s + lane) % in_len);
#pragma unroll 4
        for (int j = lane; j < out_len; j += 32) {                  // (unrolled: four loads in flight per lane)
            dst[j] = src[idx];
            idx += step;
            if (idx >= in_len) idx -= in_len;
        }
    }
}
// frame -> prefix || frame (the STS slot in front of LTS || data, :572-581)
__global__ void k_prepend(const float2 *__restrict__ prefix, int prefix_len, const float2 *__restrict__ in, float2 *__restrict__ out, long n, int len)
{
    const int out_len = prefix_len + len;
    const long total = n * out_len;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const long f = t / out_len; const int j = (int)(t - f * out_len);
        out[t] = j < prefix_len ? prefix[j] : in[f * len + (j - prefix_len)];
    }
}
}  // namespace ofdm
