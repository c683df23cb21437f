/*
 * tests/ota_oracle.c -- TEST INFRASTRUCTURE ONLY: the over-the-air path of the C driver's default mode (host/ofdm_main.c,
 * the reference's main() body) on the CPU.  It includes tests/channel_oracle.c, and through it the pinned oracle, unchanged,
 * so that Philox, the block normals and every stage are the oracle's own.  Built by tests/ota_oracle.py with the oracle's
 * flags (-O2 -ffp-contract=off).
 *
 * Flat noise layout (domain 3, k_awgn_philox_flat): Philox block b feeds samples 4b .. 4b+3 of a buffer of any length,
 * counter (frame_lo, frame_hi, b, domain), key (seed, stream).
 */
#include "channel_oracle.c"

void orc_philox_normals_flat(uint32_t seed, uint32_t stream, uint64_t frame0, long n_frames, int len, uint32_t domain, float *g)
{
    for (long f = 0; f < n_frames; ++f) {
        uint64_t fr = frame0 + (uint64_t)f;
        for (int b = 0; 4 * b < len; ++b) {
            uint32_t ctr[4] = {(uint32_t)fr, (uint32_t)(fr >> 32), (uint32_t)b, domain}, key[2] = {seed, stream}, r[4];
            float z[4];
            orc_philox4x32_10(ctr, key, r);
            block_normals(r, z);
            for (int j = 0; j < 4 && 4 * b + j < len; ++j) g[f * len + 4 * b + j] = z[j];
        }
    }
}

/* which Philox block / which of its four normals feeds sample n of an LTS||data frame (the domain layout) */
void orc_noise_slot(int n, int *blk, int *j) { noise_slot(n, blk, j); }

/* the frequency the coarse (fine = 0) or fine estimator finds, as orc_cfo_coarse / orc_cfo_fine compute it */
float orc_cfo_freq(const float *rx, int fine)
{
    const cf32 *x = (const cf32 *)rx;
    cf32 p = fine ? conj_dot(x + 192, x + 256, 64) : conj_dot(x + 80, x + 96, 16);
    double k = fine ? -1.0 / (2 * PI_REF * 64 * TS_SEC) : -1.0 / (2 * PI_REF * 16 * TS_SEC);
    return (float)(k * atan2((double)p.im, (double)p.re));
}

/* One SNR point of the driver's default mode from the repeated waveform on: flat noise g [len_rep] on the real rail at
 * snr_db (power measured on the waveform), capture window at rx_start, packet detection and selection, matched filter
 * at the selected index, coarse and fine CFO, receiver.  Returns the selected index, or -1 (nothing past selection is
 * run) when the matched filter would read past the filtered capture, where the reference's behaviour is undefined. */
int orc_ota_point(const float *rep, int len_rep, const float *g, float snr_db, int rx_start, int len_cap, const uint8_t *bits,
                  int n_sym, orc_rx_stats *st)
{
    orc_init();
    const int len = 160 + 80 * n_sym, len480 = 160 + len, n_corr = len_cap - 47;
    cf32 *ota = (cf32 *)malloc(sizeof(cf32) * (size_t)len_rep), *corr = (cf32 *)malloc(sizeof(cf32) * (size_t)n_corr);
    cf32 *rx = (cf32 *)malloc(sizeof(cf32) * (size_t)len480), *c1 = (cf32 *)malloc(sizeof(cf32) * (size_t)len480);
    cf32 *c2 = (cf32 *)malloc(sizeof(cf32) * (size_t)len480), *mod = (cf32 *)malloc(sizeof(cf32) * 48 * (size_t)n_sym);
    awgn_inject((const cf32 *)rep, g, ota, snr_db, len_rep);
    const cf32 *cap = ota + rx_start;
    orc_packet_detection((const float *)cap, len_cap, (float *)corr);
    int idx = orc_packet_selection((const float *)corr, n_corr);
    if (idx + 2 * (len480 - 1) < len_cap + 20) {
        orc_rrc_rx((const float *)cap, len_cap, idx, len480, (float *)rx);
        orc_cfo_coarse((const float *)rx, len480, (float *)c1);
        orc_cfo_fine((const float *)c1, len480, (float *)c2);
        orc_qpsk_mod(bits, n_sym, (float *)mod);
        rx_frame(c2 + 160, n_sym, bits, mod, NULL, NULL, NULL, NULL, st);
    } else {
        idx = -1;
    }
    free(ota); free(corr); free(rx); free(c1); free(c2); free(mod);
    return idx;
}
