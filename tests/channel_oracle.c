/*
 * tests/channel_oracle.c -- TEST INFRASTRUCTURE ONLY: the channels of include/ofdm_b200.h (ofdm_channel; DESIGN.md
 * "Channels") restated on the CPU.  It contains no reference code: it restates the definitions and runs them through the
 * pinned oracle's transmitter, frame power and receiver, which it includes unchanged so that their static helpers are
 * reused rather than copied.  Built by tests/channel_oracle.py with the oracle's flags (-O2 -ffp-contract=off).
 *
 *   noise 0 (real rail)  y.re = x.re + (float)(sigma * g0), y.im = x.im,          sigma = sqrt((double)np)
 *   noise 1 (complex)    y.re = x.re + (float)(sigma * g0), y.im = x.im + (float)(sigma * g1), sigma = sqrt(0.5 * (double)np)
 *   snr_def 0            np = P / (float)pow(10, snr_db/10), P the frame power of the frame on the air
 *   snr_def 1 / 2        np = (float)(1 / (64 or 128 * 10^(snr_db/10)))   (Es/N0 per data subcarrier / Eb/N0)
 * g0 = the domain-0 normal of the sample's noise slot, g1 = the normal in the same slot of domain 4.
 */
#include "../oracle/ofdm_oracle.c"

enum { DOMAIN_NOISE_Q = 4 };

/* orc_philox_normals for any domain: key (seed, stream), counter (frame_lo, frame_hi, block, domain), noise_slot layout */
void orc_philox_normals_domain(uint32_t seed, uint32_t stream, uint64_t frame0, long n_frames, int len, uint32_t domain, float *g)
{
    for (long f = 0; f < n_frames; ++f) {
        uint64_t fr = frame0 + (uint64_t)f;
        for (int n = 0; n < len; ++n) {
            int blk, j;
            noise_slot(n, &blk, &j);
            uint32_t ctr[4] = {(uint32_t)fr, (uint32_t)(fr >> 32), (uint32_t)blk, domain}, key[2] = {seed, stream}, r[4];
            float z[4];
            orc_philox4x32_10(ctr, key, r);
            block_normals(r, z);
            g[f * len + n] = z[j];
        }
    }
}

static float channel_noise_power(const cf32 *x, float snr_db, int snr_def, int len)
{
    if (snr_def == 0) {
        float snr_lin = (float)pow(10.0, (double)(snr_db / 10));
        return frame_power(x, len) / snr_lin;
    }
    double per_point = snr_def == 2 ? 128.0 : 64.0;
    return (float)(1.0 / (per_point * pow(10.0, (double)snr_db / 10.0)));
}

static void awgn_channel(const cf32 *x, const float *g0, const float *g1, cf32 *y, float snr_db, int noise, int snr_def, int len)
{
    float np = channel_noise_power(x, snr_db, snr_def, len);
    double sigma = noise ? sqrt(0.5 * (double)np) : sqrt((double)np);
    for (int i = 0; i < len; ++i) {
        y[i].re = x[i].re + (float)(sigma * (double)g0[i]);
        y[i].im = noise ? x[i].im + (float)(sigma * (double)g1[i]) : x[i].im;
    }
}

/* g1 is read only for complex noise (may be NULL otherwise) */
void orc_awgn_channel(const float *tx, const float *g0, const float *g1, float *out, float snr_db, int noise, int snr_def, int len)
{
    awgn_channel((const cf32 *)tx, g0, g1, (cf32 *)out, snr_db, noise, snr_def, len);
}

/* transmitter -> [taps, n_taps > 0] -> channel -> receiver per frame; g0, g1 [n_frames][len], taps [n_frames][n_taps][2] */
void orc_chain_channel(const uint8_t *bits, const float *g0, const float *g1, const float *taps, int n_taps, long n_frames, int n_sym,
                       float snr_db, int noise, int snr_def, orc_counters *acc, int *frame_bit_errors, float *frame_evm_lin)
{
    orc_init();
    int len = 160 + 80 * n_sym;
    cf32 *tx = (cf32 *)malloc(sizeof(cf32) * (size_t)len), *ch = (cf32 *)malloc(sizeof(cf32) * (size_t)len);
    cf32 *ota = (cf32 *)malloc(sizeof(cf32) * (size_t)len), *mod = (cf32 *)malloc(sizeof(cf32) * 48 * (size_t)n_sym);
    for (long f = 0; f < n_frames; ++f) {
        const uint8_t *b = bits + f * 96 * n_sym;
        tx_frame(b, n_sym, tx, mod);
        const cf32 *air = tx;
        if (n_taps > 0) {
            orc_apply_taps((const float *)tx, taps + f * n_taps * 2, n_taps, (float *)ch, len);
            air = ch;
        }
        awgn_channel(air, g0 + f * len, g1 ? g1 + f * len : NULL, ota, snr_db, noise, snr_def, len);
        orc_rx_stats st;
        rx_frame(ota, n_sym, b, mod, NULL, NULL, NULL, NULL, &st);
        accumulate(acc, &st, n_sym);
        if (frame_bit_errors) frame_bit_errors[f] = st.bit_errors;
        if (frame_evm_lin) frame_evm_lin[f] = st.evm_lin;
    }
    free(tx); free(ch); free(ota); free(mod);
}
