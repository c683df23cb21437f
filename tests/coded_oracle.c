/*
 * tests/coded_oracle.c -- TEST INFRASTRUCTURE ONLY: the coded link of include/ofdm_b200.h (ofdm_code; DESIGN.md section 6.2)
 * restated on the CPU from its definitions.  It includes the channel oracle (and through it the pinned oracle, unchanged) so that
 * the transmitter, the channels and the receiver are theirs.  Built by tests/coded_oracle.py with the oracle's flags
 * (-O2 -ffp-contract=off): every float operation below rounds once, as the GPU's __fmul_rn / __fadd_rn do.
 *
 *   encoder   K = 7, A = parity(W & 0133), B = parity(W & 0171), W = 7-bit window, bit 6 = newest input bit; starts in state 0
 *   frame     K_info = n_sym N_DBPS - 6 information bits (bits 0 .. K_info-1 of the frame's packed words), then 6 zero tail bits
 *   rate 3/4  of A0 B0 A1 B1 A2 B2 send A0 B0 A1 B2
 *   interleave coded bit k of a symbol -> position i = 6 (k mod 16) + k / 16; data point i >> 1, I rail if i even, Q if odd
 *   precode   payload bits (2d, 2d+1) = (!c1, c0 ^ c1), c0 / c1 the coded bits on the I / Q rail of data point d
 *   decoder   inputs L (soft w eq, w = |H|^2; hard +-1, 0 and NaN negative; non-finite L = 0), metric sum L (2c - 1) in float,
 *             new metric of state t = max over its predecessors 2(t mod 32) and 2(t mod 32) + 1 (the higher one only if strictly
 *             larger), then every metric minus the new metric of state 0; start and end in state 0
 */
#include "channel_oracle.c"

static int dbps(int rate) { return rate == 1 ? 48 : 72; }
static int parity7(unsigned v) { v &= 127u; v ^= v >> 4; v ^= v >> 2; v ^= v >> 1; return (int)(v & 1u); }
int orc_interleave(int k) { return 6 * (k % 16) + k / 16; }

/* one frame: info bits (one byte per bit, K_info of them) -> payload bits [96 n_sym] */
void orc_conv_encode(int rate, const uint8_t *info, int n_sym, uint8_t *payload)
{
    const int N = dbps(rate), T = n_sym * N, k_info = T - 6;
    uint8_t *coded = (uint8_t *)malloc((size_t)(2 * T));
    int n_coded = 0;
    unsigned w = 0;
    for (int n = 0; n < T; ++n) {
        const unsigned x = n < k_info ? info[n] & 1u : 0u;
        w = (w >> 1) | (x << 6);
        const uint8_t a = (uint8_t)parity7(w & 0133u), b = (uint8_t)parity7(w & 0171u);
        if (rate == 1 || n % 3 == 0) { coded[n_coded++] = a; coded[n_coded++] = b; }
        else if (n % 3 == 1) coded[n_coded++] = a;
        else coded[n_coded++] = b;
    }
    for (int s = 0; s < n_sym; ++s) {
        uint8_t pos[96];
        for (int k = 0; k < 96; ++k) pos[orc_interleave(k)] = coded[96 * s + k];
        for (int d = 0; d < 48; ++d) {
            const uint8_t c0 = pos[2 * d], c1 = pos[2 * d + 1];
            payload[96 * s + 2 * d] = (uint8_t)!c1;
            payload[96 * s + 2 * d + 1] = (uint8_t)(c0 ^ c1);
        }
    }
    free(coded);
}

/* one frame: H [64] centred, eq [n_sym * 48] -> decoded information bits [K_info] */
void orc_viterbi(int rate, int decision, const float *H_f, const float *eq_f, int n_sym, uint8_t *out)
{
    orc_init();
    const cf32 *H = (const cf32 *)H_f, *eq = (const cf32 *)eq_f;
    const int N = dbps(rate), T = n_sym * N, k_info = T - 6;
    int centred_of[48];
    for (int c = 0; c < 64; ++c) if (data_index_of[c] >= 0) centred_of[data_index_of[c]] = c;
    float *La = (float *)malloc(sizeof(float) * (size_t)T), *Lb = (float *)malloc(sizeof(float) * (size_t)T);
    for (int s = 0; s < n_sym; ++s) {
        float Li[96], Lk[96];
        for (int i = 0; i < 96; ++i) {
            const int d = i >> 1;
            const cf32 h = H[centred_of[d]], e = eq[48 * s + d];
            const float v = (i & 1) ? e.im : e.re;
            float L;
            if (decision == 1) L = v > 0.0f ? 1.0f : -1.0f;
            else {
                const float w = h.re * h.re + h.im * h.im;
                L = w * v;
            }
            Li[i] = isfinite(L) ? L : 0.0f;
        }
        for (int k = 0; k < 96; ++k) Lk[k] = Li[orc_interleave(k)];
        for (int j = 0; j < N; ++j) {
            const int n = s * N + j;
            if (rate == 1) { La[n] = Lk[2 * j]; Lb[n] = Lk[2 * j + 1]; continue; }
            const int g = j / 3, r = j % 3;
            La[n] = r == 2 ? 0.0f : Lk[4 * g + (r == 0 ? 0 : 2)];
            Lb[n] = r == 1 ? 0.0f : Lk[4 * g + (r == 0 ? 1 : 3)];
        }
    }
    float M[64], Mn[64];
    uint8_t *surv = (uint8_t *)malloc((size_t)T * 64);
    for (int t = 0; t < 64; ++t) M[t] = t == 0 ? 0.0f : -INFINITY;
    for (int n = 0; n < T; ++n) {
        for (int t = 0; t < 64; ++t) {
            const unsigned b = (unsigned)t >> 5;
            float cand[2];
            for (int e = 0; e < 2; ++e) {
                const unsigned s = (((unsigned)t << 1) & 63u) | (unsigned)e, W = (b << 6) | s;
                const float bm = (float)(2 * parity7(W & 0133u) - 1) * La[n] + (float)(2 * parity7(W & 0171u) - 1) * Lb[n];
                cand[e] = M[s] + bm;
            }
            const int dec = cand[1] > cand[0];
            Mn[t] = cand[dec];
            surv[(size_t)n * 64 + t] = (uint8_t)dec;
        }
        const float z = Mn[0];
        for (int t = 0; t < 64; ++t) M[t] = Mn[t] - z;
    }
    int state = 0;
    for (int n = T - 1; n >= 0; --n) {
        if (n < k_info) out[n] = (uint8_t)(state >> 5);
        state = ((state << 1) & 63) | surv[(size_t)n * 64 + state];
    }
    free(La); free(Lb); free(surv);
}

/* the coded chain per frame: encoder -> transmitter -> [taps] -> channel (Eb/N0 per information bit) -> receiver (raw counters,
 * H and eq) -> decoder (coded counters).  info [n_frames][96 n_sym] one byte per bit (bits >= K_info unused). */
void orc_coded_chain(int rate, int decision, const uint8_t *info, const float *g0, const float *g1, const float *taps, int n_taps,
                     long n_frames, int n_sym, float snr_db, int noise, int snr_def, orc_counters *coded_acc, orc_counters *raw_acc)
{
    orc_init();
    const int len = 160 + 80 * n_sym, k_info = n_sym * dbps(rate) - 6;
    cf32 *tx = (cf32 *)malloc(sizeof(cf32) * (size_t)len), *ch = (cf32 *)malloc(sizeof(cf32) * (size_t)len);
    cf32 *ota = (cf32 *)malloc(sizeof(cf32) * (size_t)len), *mod = (cf32 *)malloc(sizeof(cf32) * 48 * (size_t)n_sym);
    cf32 *eq = (cf32 *)malloc(sizeof(cf32) * 48 * (size_t)n_sym), H[64];
    uint8_t *payload = (uint8_t *)malloc((size_t)(96 * n_sym)), *dec = (uint8_t *)malloc((size_t)k_info);
    for (long f = 0; f < n_frames; ++f) {
        const uint8_t *b = info + f * 96 * n_sym;
        orc_conv_encode(rate, b, n_sym, payload);
        tx_frame(payload, n_sym, tx, mod);
        const cf32 *air = tx;
        if (n_taps > 0) {
            orc_apply_taps((const float *)tx, taps + f * n_taps * 2, n_taps, (float *)ch, len);
            air = ch;
        }
        const float *n0 = g0 + f * len, *n1 = g1 ? g1 + f * len : NULL;
        if (snr_def == 2) {                   /* Eb/N0 of the information bits: np = 1 / (64 2R 10^(snr/10)) */
            const double per_point = 64.0 * (rate == 1 ? 1.0 : 1.5);
            const float np = (float)(1.0 / (per_point * pow(10.0, (double)snr_db / 10.0)));
            const double sigma = noise ? sqrt(0.5 * (double)np) : sqrt((double)np);
            for (int i = 0; i < len; ++i) {
                ota[i].re = air[i].re + (float)(sigma * (double)n0[i]);
                ota[i].im = noise ? air[i].im + (float)(sigma * (double)n1[i]) : air[i].im;
            }
        } else {
            awgn_channel(air, n0, n1, ota, snr_db, noise, snr_def, len);
        }
        orc_rx_stats st;
        rx_frame(ota, n_sym, payload, mod, H, eq, NULL, NULL, &st);
        accumulate(raw_acc, &st, n_sym);
        orc_viterbi(rate, decision, (const float *)H, (const float *)eq, n_sym, dec);
        uint64_t e = 0;
        for (int j = 0; j < k_info; ++j) e += dec[j] != b[j];
        coded_acc->bit_errors += e;
        coded_acc->bits += (uint64_t)k_info;
        coded_acc->frames_in_error += e > 0;
        coded_acc->frames += 1;
    }
    free(tx); free(ch); free(ota); free(mod); free(eq); free(payload); free(dec);
}
