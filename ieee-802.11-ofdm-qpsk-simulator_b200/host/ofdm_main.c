/*
 * ofdm_main.c -- C host driver over the C-ABI (include/ofdm_b200.h): the batched counterpart of the
 * reference's main() (OFDM.c:1187-1236).  Same sweep (default 35 points, 6..40 dB, OFDM.c:18,1197), same
 * four result files in the same format (write_float_array_to_file, OFDM.c:123-143, 1228-1231) so that
 * scripts/OFDM_Plotting.py of the reference reads them unchanged:
 *     <outdir>/Output_SNR.txt          SNR points
 *     <outdir>/Output_EVM_AGC.txt      EVM *before* the slicer, dB   (the reference's naming, OFDM.c:1229)
 *     <outdir>/Output_EVM_AGC_DB.txt   EVM after the slicer, dB      (OFDM.c:1230)
 *     <outdir>/Output_BER.txt          BER
 * Two payload sources:
 *   --message TEXT (default "Hey! I am Vivaswan", OFDM.c:20): Data_Generator's codec (OFDM.c:435-465,
 *       MSB-first ASCII bits, space-padded to a multiple of 96 bits), one frame, prints the received
 *       message per SNR point like Receiver() does (OFDM.c:1169-1182).  By default this mode runs the
 *       reference's WHOLE over-the-air path (STS, x2 + RRC, x10 repetition, noise on the repeated waveform,
 *       random capture window, packet detection / selection, matched filter + decimation, coarse + fine CFO,
 *       then the stage chain), OFDM.c:467-618 and :941-1165; --stage-chain keeps only the stage chain;
 *   --frames N (N > 1): N frames of Philox random bits per SNR point through the fused Monte-Carlo kernel.
 *   --taps L (with --frames N): configs[4], per-frame random multipath channel with L <= 16 taps in front of the noise;
 *   --target-errors E [--max-bits B] [--round-frames R]: configs[3] as BASELINE.json states it -- every SNR point runs until it
 *       has >= E bit errors or >= B bits (default B = E / 1e-7: the BER-1e-7 budget), in rounds of R frames (default 4 Mi);
 *       finished points leave the kernel's SNR list, the others keep their noise streams.  With --gpus N every round's frame
 *       range is split across the GPUs (so the slow high-SNR points use all of them) and the round's counters are all-reduced
 *       before the stop decisions -- summed on the host by default (this is one process driving every GPU; the partial counters are a
 *       few hundred bytes), or with NCCL all-reduces (--round-reduce-nccl): the result does not depend on the GPU count;
 *   --draws FILE [--bits FILE]: configs[1] from C -- injected-noise sweep (ofdm_sweep_inject_host): FILE holds one float32
 *       standard-normal draw per sample, [frames][160 + 80 nsym] (e.g. the reference's captured g_keep stream); the payload is
 *       the Philox bit stream of --seed, or packed uint32 words [frames][3 nsym] from --bits;
 *   --noise real|complex, --snr-def frame_power|esn0|ebn0 (with --frames N or --target-errors E, also with --taps and --gpus): the
 *       channel of the Monte-Carlo sweep (ofdm_channel, include/ofdm_b200.h).  The default, real / frame_power, is the reference's:
 *       noise on the I rail only, SNR = measured frame power / noise power.  complex = circular complex noise, half of the noise
 *       power per rail; esn0 / ebn0 = Es/N0 per data subcarrier / Eb/N0, the SNR axis of textbook QPSK curves.  Not available
 *       with --message or --draws, whose channels are the reference's by definition;
 *   --gpus N: the frames of the Monte-Carlo sweep are sharded across N GPUs of this node by global frame index
 *       (one context per GPU, all driven from this thread) and the counters are summed with ONE NCCL all-reduce
 *       per buffer type (built with -DOFDM_WITH_NCCL; link -lnccl).
 * There is no CPU fallback: without a CUDA device the program exits with an error.
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "ofdm_b200.h"
#ifdef OFDM_WITH_NCCL
#include <nccl.h>
#endif

#define CHECK(call)                                                                                  \
    do {                                                                                             \
        int st_ = (call);                                                                            \
        if (st_ != OFDM_OK) {                                                                        \
            fprintf(stderr, "%s failed: %s (%s)\n", #call, ofdm_strerror(st_), ctx ? ofdm_last_error(ctx) : ""); \
            return 1;                                                                                \
        }                                                                                            \
    } while (0)

/* Data_Generator + Decimal_To_Binary, OFDM.c:401-465: 8 bits per character, MSB first, padded with ' ' */
static int encode_message(const char *msg, uint8_t **bits_out, int *n_sym_out)
{
    int len = (int)strlen(msg);
    int n_sym = (int)ceil(8 * len / 96.0);
    if (n_sym < 1) n_sym = 1;
    int total_bits = n_sym * 96, total_chars = total_bits / 8;
    uint8_t *bits = (uint8_t *)calloc((size_t)total_bits, 1);
    if (!bits) return OFDM_ERR_NOMEM;
    for (int i = 0; i < total_chars; ++i) {
        int ch = i < len ? (unsigned char)msg[i] : ' ';
        for (int j = 0; j < 8; ++j) bits[8 * i + j] = (uint8_t)((ch >> (7 - j)) & 1);
    }
    *bits_out = bits; *n_sym_out = n_sym;
    return OFDM_OK;
}

static void pack_bits(const uint8_t *bits, int n_bits, uint32_t *words)
{
    memset(words, 0, (size_t)(n_bits / 32) * sizeof(uint32_t));
    for (int j = 0; j < n_bits; ++j) words[j >> 5] |= (uint32_t)(bits[j] & 1u) << (j & 31);
}

/* Message_Generator + Binary_To_Decimal, OFDM.c:910-939 */
static void decode_message(const uint32_t *words, int n_bits, char *out)
{
    for (int i = 0; i < n_bits / 8; ++i) {
        int v = 0;
        for (int j = 0; j < 8; ++j) { int b = 8 * i + j; v = v * 2 + (int)((words[b >> 5] >> (b & 31)) & 1u); }
        out[i] = (char)v;
    }
    out[n_bits / 8] = 0;
}

static double now_s(void)
{
    struct timespec t;
    clock_gettime(CLOCK_MONOTONIC, &t);
    return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec;
}
static void report_rate(const char *what, int n_gpus, long frames, int n_sym, int n_snr, double seconds)
{
    fprintf(stderr, "%s: %ld frames x %d symbols x %d SNR points on %d GPU(s) in %.3f s = %.3e data symbols/s\n", what, frames, n_sym,
            n_snr, n_gpus, seconds, (double)frames * n_sym * n_snr / seconds);
}

#ifdef OFDM_WITH_NCCL
#define NCHECK(call)                                                                   \
    do {                                                                               \
        ncclResult_t r_ = (call);                                                      \
        if (r_ != ncclSuccess) { fprintf(stderr, "%s failed: %s\n", #call, ncclGetErrorString(r_)); return 1; } \
    } while (0)

/* SURVEY 8(e): shard (frame range) across GPUs, counter-based RNG keyed on the global frame index, one all-reduce */
static int sweep_multi_gpu(int n_gpus, unsigned seed, long frames, int n_sym, const ofdm_channel *ch, const float *SNR, int n_snr, int mode,
                           ofdm_counters *totals, unsigned long long target_errors, unsigned long long max_bits, long round_frames, int round_reduce_host)
{
    const int n_taps = ch->n_taps;
    ofdm_ctx *ctxs[8] = {0};
    ofdm_ctx *ctx = NULL;
    void *cnt[8], *ints[8], *dbls[8];
    ncclComm_t comms[8];
    int devs[8];
    if (n_gpus < 1 || n_gpus > 8) { fprintf(stderr, "--gpus must be 1..8\n"); return 2; }
    for (int d = 0; d < n_gpus; ++d) {
        devs[d] = d;
        CHECK(ofdm_ctx_create(&ctxs[d], d));
        ctx = ctxs[d];
        CHECK(ofdm_dev_alloc(ctx, &cnt[d], sizeof(ofdm_counters) * (size_t)n_snr));
        CHECK(ofdm_dev_alloc(ctx, &ints[d], sizeof(uint64_t) * 5 * (size_t)n_snr));
        CHECK(ofdm_dev_alloc(ctx, &dbls[d], sizeof(double) * 3 * (size_t)n_snr));
        CHECK(ofdm_memset_dev(ctx, cnt[d], 0, sizeof(ofdm_counters) * (size_t)n_snr));
    }
    NCHECK(ncclCommInitAll(comms, n_gpus, devs));
    for (int d = 0; d < n_gpus; ++d) {                      /* first use of a kernel on a device loads it: keep that out of the timing */
        ctx = ctxs[d];
        CHECK(ofdm_mc_sweep_channel_dev(ctx, ch, seed, 0, 256, n_sym, SNR, NULL, n_snr, mode, (ofdm_counters *)cnt[d]));
        CHECK(ofdm_memset_dev(ctx, cnt[d], 0, sizeof(ofdm_counters) * (size_t)n_snr));
        CHECK(ofdm_counters_pack(ctx, (const ofdm_counters *)cnt[d], n_snr, (uint64_t *)ints[d], (double *)dbls[d]));
        CHECK(ofdm_ctx_sync(ctx));
    }
    /* ... and so does the first collective of a communicator (NCCL connects its peers lazily: ~0.1 s on 8 GPUs): one all-reduce
     * of the zeroed buffers before the clock starts */
    NCHECK(ncclGroupStart());
    for (int d = 0; d < n_gpus; ++d) {
        NCHECK(ncclAllReduce(ints[d], ints[d], 5 * (size_t)n_snr, ncclUint64, ncclSum, comms[d], (cudaStream_t)ofdm_ctx_stream(ctxs[d])));
        NCHECK(ncclAllReduce(dbls[d], dbls[d], 3 * (size_t)n_snr, ncclDouble, ncclSum, comms[d], (cudaStream_t)ofdm_ctx_stream(ctxs[d])));
    }
    NCHECK(ncclGroupEnd());
    for (int d = 0; d < n_gpus; ++d) { ctx = ctxs[d]; CHECK(ofdm_ctx_sync(ctx)); }
    if (target_errors > 0) {
        /* configs[3]'s stop rule, sharded as (SNR point x frame range): every GPU works on every still-active point, on its
         * slice of the round's frames; one all-reduce per buffer type per round; identical stop decisions everywhere */
        int active[64], n_active = n_snr, rounds = 0;
        unsigned long long done_frames = 0;
        ofdm_counters part[64];
        memset(totals, 0, sizeof(ofdm_counters) * (size_t)n_snr);
        for (int i = 0; i < n_snr; ++i) active[i] = i;
        const double t0 = now_s();
        while (n_active > 0) {
            float snr_a[64]; uint32_t stream_a[64];
            for (int j = 0; j < n_active; ++j) { snr_a[j] = SNR[active[j]]; stream_a[j] = (uint32_t)active[j]; }
            for (int d = 0; d < n_gpus; ++d) {
                long base = round_frames / n_gpus, rem = round_frames % n_gpus;
                long lo = d * base + (d < rem ? d : rem), n = base + (d < rem ? 1 : 0);
                ctx = ctxs[d];
                CHECK(ofdm_memset_dev(ctx, cnt[d], 0, sizeof(ofdm_counters) * (size_t)n_active));
                CHECK(ofdm_mc_sweep_channel_dev(ctx, ch, seed, (uint64_t)rounds * (uint64_t)round_frames + (uint64_t)lo, n, n_sym, snr_a, stream_a,
                                                n_active, mode, (ofdm_counters *)cnt[d]));
                if (!round_reduce_host) CHECK(ofdm_counters_pack(ctx, (const ofdm_counters *)cnt[d], n_active, (uint64_t *)ints[d], (double *)dbls[d]));
            }
            if (round_reduce_host) {
                /* one process drives every GPU: the round's partial counters (a few hundred bytes per GPU) can also be summed on the host */
                static ofdm_counters per_gpu[8][64];
                for (int d = 0; d < n_gpus; ++d) { ctx = ctxs[d]; CHECK(ofdm_memcpy_d2h(ctx, per_gpu[d], cnt[d], sizeof(ofdm_counters) * (size_t)n_active)); }
                for (int d = 0; d < n_gpus; ++d) { ctx = ctxs[d]; CHECK(ofdm_ctx_sync(ctx)); }
                memset(part, 0, sizeof part);
                for (int d = 0; d < n_gpus; ++d)
                    for (int j = 0; j < n_active; ++j) {
                        part[j].bit_errors += per_gpu[d][j].bit_errors; part[j].bits += per_gpu[d][j].bits; part[j].frames_in_error += per_gpu[d][j].frames_in_error;
                        part[j].rail_errors += per_gpu[d][j].rail_errors; part[j].frames += per_gpu[d][j].frames;
                        part[j].sum_err2 += per_gpu[d][j].sum_err2; part[j].sum_ref2 += per_gpu[d][j].sum_ref2; part[j].sum_evm_lin += per_gpu[d][j].sum_evm_lin;
                    }
            } else {
                NCHECK(ncclGroupStart());
                for (int d = 0; d < n_gpus; ++d) {
                    NCHECK(ncclAllReduce(ints[d], ints[d], 5 * (size_t)n_active, ncclUint64, ncclSum, comms[d], (cudaStream_t)ofdm_ctx_stream(ctxs[d])));
                    NCHECK(ncclAllReduce(dbls[d], dbls[d], 3 * (size_t)n_active, ncclDouble, ncclSum, comms[d], (cudaStream_t)ofdm_ctx_stream(ctxs[d])));
                }
                NCHECK(ncclGroupEnd());
                ctx = ctxs[0];
                CHECK(ofdm_counters_unpack(ctx, (ofdm_counters *)cnt[0], n_active, (const uint64_t *)ints[0], (const double *)dbls[0]));
                CHECK(ofdm_memcpy_d2h(ctx, part, cnt[0], sizeof(ofdm_counters) * (size_t)n_active));
                for (int d = 0; d < n_gpus; ++d) { ctx = ctxs[d]; CHECK(ofdm_ctx_sync(ctx)); }
            }
            int keep = 0;
            for (int j = 0; j < n_active; ++j) {
                ofdm_counters *t = &totals[active[j]];
                t->bit_errors += part[j].bit_errors; t->bits += part[j].bits; t->frames_in_error += part[j].frames_in_error;
                t->rail_errors += part[j].rail_errors; t->frames += part[j].frames;
                t->sum_err2 += part[j].sum_err2; t->sum_ref2 += part[j].sum_ref2; t->sum_evm_lin += part[j].sum_evm_lin;
                done_frames += part[j].frames;
                if (t->bit_errors < target_errors && t->bits < max_bits) active[keep++] = active[j];
            }
            n_active = keep;
            ++rounds;
        }
        const double dt = now_s() - t0;
        fprintf(stderr, "until-sweep: %d rounds of %ld frames, %llu frame-points x %d symbols on %d GPU(s) in %.3f s = %.3e data symbols/s (round totals: %s)\n", rounds,
                round_frames, done_frames, n_sym, n_gpus, dt, (double)done_frames * n_sym / dt, round_reduce_host ? "summed on the host" : "NCCL all-reduce");
        for (int d = 0; d < n_gpus; ++d) {
            ncclCommDestroy(comms[d]);
            ofdm_dev_free(ctxs[d], cnt[d]); ofdm_dev_free(ctxs[d], ints[d]); ofdm_dev_free(ctxs[d], dbls[d]);
            ofdm_ctx_destroy(ctxs[d]);
        }
        return 0;
    }
    const double t0 = now_s();
    for (int d = 0; d < n_gpus; ++d) {                      /* all GPUs run their shard concurrently (async launches) */
        long base = frames / n_gpus, rem = frames % n_gpus;
        long lo = d * base + (d < rem ? d : rem), n = base + (d < rem ? 1 : 0);
        ctx = ctxs[d];
        CHECK(ofdm_mc_sweep_channel_dev(ctx, ch, seed, (uint64_t)lo, n, n_sym, SNR, NULL, n_snr, mode, (ofdm_counters *)cnt[d]));
        CHECK(ofdm_counters_pack(ctx, (const ofdm_counters *)cnt[d], n_snr, (uint64_t *)ints[d], (double *)dbls[d]));
    }
    NCHECK(ncclGroupStart());
    for (int d = 0; d < n_gpus; ++d) {
        NCHECK(ncclAllReduce(ints[d], ints[d], 5 * (size_t)n_snr, ncclUint64, ncclSum, comms[d], (cudaStream_t)ofdm_ctx_stream(ctxs[d])));
        NCHECK(ncclAllReduce(dbls[d], dbls[d], 3 * (size_t)n_snr, ncclDouble, ncclSum, comms[d], (cudaStream_t)ofdm_ctx_stream(ctxs[d])));
    }
    NCHECK(ncclGroupEnd());
    for (int d = 0; d < n_gpus; ++d) {
        ctx = ctxs[d];
        CHECK(ofdm_counters_unpack(ctx, (ofdm_counters *)cnt[d], n_snr, (const uint64_t *)ints[d], (const double *)dbls[d]));
    }
    ctx = ctxs[0];
    CHECK(ofdm_memcpy_d2h(ctx, totals, cnt[0], sizeof(ofdm_counters) * (size_t)n_snr));
    for (int d = 0; d < n_gpus; ++d) { ctx = ctxs[d]; CHECK(ofdm_ctx_sync(ctx)); }
    report_rate(n_taps > 0 ? "multipath sweep" : "sweep", n_gpus, frames, n_sym, n_snr, now_s() - t0);
    for (int d = 0; d < n_gpus; ++d) {
        ncclCommDestroy(comms[d]);
        ofdm_dev_free(ctxs[d], cnt[d]); ofdm_dev_free(ctxs[d], ints[d]); ofdm_dev_free(ctxs[d], dbls[d]);
        ofdm_ctx_destroy(ctxs[d]);
    }
    return 0;
}
#endif

int main(int argc, char **argv)
{
    const char *message = "Hey! I am Vivaswan";          /* OFDM.c:20 */
    const char *outdir = "data", *dump = NULL;
    long frames = 1;
    int n_sym = 2, n_snr = 35, device = 0, mode = OFDM_MODE_EXACT, quiet = 0, n_gpus = 1, full_chain = 1, n_taps = 0;
    float snr_start = 6.0f, snr_step = 1.0f;             /* OFDM.c:18, :1195-1198 */
    unsigned seed = 1;
    unsigned long long target_errors = 0, max_bits = 0;
    long round_frames = 1L << 22;
    const char *draws_file = NULL, *bits_file = NULL;
    ofdm_channel ch = {OFDM_NOISE_REAL_RAIL, OFDM_SNR_FRAME_POWER, 0};
    int channel_set = 0;                 /* --noise / --snr-def given */
    int round_reduce_host = 1;           /* until rule: per-round totals summed on the host (measured 8 GPUs, 13 rounds: 0.033 s against 0.294 s with two
                                            single-process NCCL group all-reduces per round, profiles/r2_c_driver_until_8gpu.txt) */
    for (int i = 1; i < argc; ++i) {
        const char *a = argv[i], *v = i + 1 < argc ? argv[i + 1] : NULL;
        if (!strcmp(a, "--quiet")) { quiet = 1; continue; }
        if (!strcmp(a, "--stage-chain")) { full_chain = 0; continue; }
        if (!strcmp(a, "--full-chain")) { full_chain = 1; continue; }
        if (!strcmp(a, "--round-reduce-host")) { round_reduce_host = 1; continue; }
        if (!strcmp(a, "--round-reduce-nccl")) { round_reduce_host = 0; continue; }
        if (!v) { fprintf(stderr, "missing value for %s\n", a); return 2; }
        if (!strcmp(a, "--message")) message = v;
        else if (!strcmp(a, "--frames")) frames = atol(v);
        else if (!strcmp(a, "--nsym")) n_sym = atoi(v);
        else if (!strcmp(a, "--snr-start")) snr_start = (float)atof(v);
        else if (!strcmp(a, "--snr-step")) snr_step = (float)atof(v);
        else if (!strcmp(a, "--snr-count")) n_snr = atoi(v);
        else if (!strcmp(a, "--seed")) seed = (unsigned)strtoul(v, NULL, 10);
        else if (!strcmp(a, "--device")) device = atoi(v);
        else if (!strcmp(a, "--gpus")) n_gpus = atoi(v);
        else if (!strcmp(a, "--taps")) n_taps = atoi(v);
        else if (!strcmp(a, "--target-errors")) target_errors = strtoull(v, NULL, 10);
        else if (!strcmp(a, "--max-bits")) max_bits = strtoull(v, NULL, 10);
        else if (!strcmp(a, "--round-frames")) round_frames = atol(v);
        else if (!strcmp(a, "--draws")) draws_file = v;
        else if (!strcmp(a, "--bits")) bits_file = v;
        else if (!strcmp(a, "--outdir")) outdir = v;
        else if (!strcmp(a, "--dump")) dump = v;
        else if (!strcmp(a, "--mode")) mode = !strcmp(v, "fast") ? OFDM_MODE_FAST : OFDM_MODE_EXACT;
        else if (!strcmp(a, "--noise")) {
            if (!strcmp(v, "real")) ch.noise = OFDM_NOISE_REAL_RAIL;
            else if (!strcmp(v, "complex")) ch.noise = OFDM_NOISE_COMPLEX;
            else { fprintf(stderr, "--noise must be real or complex\n"); return 2; }
            channel_set = 1;
        } else if (!strcmp(a, "--snr-def")) {
            if (!strcmp(v, "frame_power")) ch.snr_def = OFDM_SNR_FRAME_POWER;
            else if (!strcmp(v, "esn0")) ch.snr_def = OFDM_SNR_ESN0;
            else if (!strcmp(v, "ebn0")) ch.snr_def = OFDM_SNR_EBN0;
            else { fprintf(stderr, "--snr-def must be frame_power, esn0 or ebn0\n"); return 2; }
            channel_set = 1;
        }
        else { fprintf(stderr, "unknown option %s\n", a); return 2; }
        ++i;
    }
    if (n_snr < 1 || n_snr > 64 || frames < 1) { fprintf(stderr, "need 1 <= snr-count <= 64 and frames >= 1\n"); return 2; }
    if (target_errors > 0 && max_bits == 0) max_bits = target_errors * 10000000ULL;        /* the BER-1e-7 budget */
    if (round_frames < 1) { fprintf(stderr, "--round-frames must be >= 1\n"); return 2; }
    if (channel_set && (draws_file || (frames < 2 && target_errors == 0))) {
        fprintf(stderr, "--noise / --snr-def choose the channel of the Monte-Carlo sweeps (--frames N > 1 or --target-errors E); "
                        "--message and --draws run the reference's channel\n");
        return 2;
    }
    ch.n_taps = n_taps;
    const int reference_channel = ch.noise == OFDM_NOISE_REAL_RAIL && ch.snr_def == OFDM_SNR_FRAME_POWER;

    ofdm_ctx *ctx = NULL;
    float SNR[64], EVM_dB[64], EVM_AGC_dB[64], BER[64];
    for (int i = 0; i < n_snr; ++i) SNR[i] = snr_start + snr_step * (float)i;
    ofdm_counters totals[64];

    if (n_gpus > 1) {
#ifdef OFDM_WITH_NCCL
        if (frames < 2 && target_errors == 0) { fprintf(stderr, "--gpus needs --frames N > 1 or --target-errors E\n"); return 2; }
        int rc = sweep_multi_gpu(n_gpus, seed, frames, n_sym, &ch, SNR, n_snr, mode, totals, target_errors, max_bits, round_frames, round_reduce_host);
        if (rc) return rc;
#else
        fprintf(stderr, "built without NCCL (make ofdm_sweep NCCL=1)\n");
        return 2;
#endif
    }
    if (n_gpus <= 1) CHECK(ofdm_ctx_create(&ctx, device));

    if (n_gpus > 1) {
        /* totals already hold the all-reduced counters */
    } else if (draws_file) {                           /* configs[1]: injected-noise sweep from host buffers */
        const int len = OFDM_FRAME_LEN(n_sym);
        FILE *fd = fopen(draws_file, "rb");
        if (!fd) { perror(draws_file); return 1; }
        fseek(fd, 0, SEEK_END);
        const long n_avail = ftell(fd) / ((long)len * 4);
        fseek(fd, 0, SEEK_SET);
        if (frames <= 1 || frames > n_avail) frames = n_avail;
        if (frames < 1) { fprintf(stderr, "%s: shorter than one frame of draws (%d floats)\n", draws_file, len); return 1; }
        void *g_host = NULL, *b_host = NULL;
        CHECK(ofdm_host_alloc(ctx, &g_host, (size_t)frames * len * 4));
        CHECK(ofdm_host_alloc(ctx, &b_host, (size_t)frames * n_sym * 12));
        if (fread(g_host, (size_t)len * 4, (size_t)frames, fd) != (size_t)frames) { fprintf(stderr, "%s: short read\n", draws_file); return 1; }
        fclose(fd);
        if (bits_file) {
            FILE *fb = fopen(bits_file, "rb");
            if (!fb) { perror(bits_file); return 1; }
            if (fread(b_host, (size_t)n_sym * 12, (size_t)frames, fb) != (size_t)frames) { fprintf(stderr, "%s: short read\n", bits_file); return 1; }
            fclose(fb);
        } else {                                       /* the Philox bit stream of --seed (frame index = position in the file) */
            void *d_b = NULL;
            CHECK(ofdm_dev_alloc(ctx, &d_b, (size_t)frames * n_sym * 12));
            CHECK(ofdm_random_bits(ctx, seed, 0, frames, n_sym, (uint32_t *)d_b));
            CHECK(ofdm_memcpy_d2h(ctx, b_host, d_b, (size_t)frames * n_sym * 12));
            CHECK(ofdm_ctx_sync(ctx));
            ofdm_dev_free(ctx, d_b);
        }
        const double t0 = now_s();
        CHECK(ofdm_sweep_inject_host(ctx, (const uint32_t *)b_host, (const float *)g_host, frames, n_sym, SNR, n_snr, mode, totals));
        report_rate("injected-noise sweep (host buffers)", 1, frames, n_sym, n_snr, now_s() - t0);
        ofdm_host_free(ctx, g_host); ofdm_host_free(ctx, b_host);
    } else if (target_errors > 0) {                    /* configs[3]: until >= E errors or the bit budget, one GPU */
        int rounds = 0;
        const double t0 = now_s();
        CHECK(ofdm_mc_sweep_channel_until(ctx, &ch, seed, 0, n_sym, SNR, n_snr, mode, target_errors, max_bits, round_frames, totals, &rounds));
        unsigned long long fp = 0;
        for (int i = 0; i < n_snr; ++i) fp += totals[i].frames;
        const double dt = now_s() - t0;
        fprintf(stderr, "until-sweep: %d rounds of %ld frames, %llu frame-points x %d symbols on 1 GPU(s) in %.3f s = %.3e data symbols/s\n", rounds, round_frames,
                fp, n_sym, dt, (double)fp * n_sym / dt);
    } else if (frames > 1) {                           /* Monte-Carlo sweep through the channel; --taps: configs[4]'s multipath taps */
        void *d_cnt = NULL;
        CHECK(ofdm_dev_alloc(ctx, &d_cnt, sizeof(ofdm_counters) * (size_t)n_snr));
        CHECK(ofdm_memset_dev(ctx, d_cnt, 0, sizeof(ofdm_counters) * (size_t)n_snr));
        const double t0 = now_s();
        CHECK(ofdm_mc_sweep_channel_dev(ctx, &ch, seed, 0, frames, n_sym, SNR, NULL, n_snr, mode, (ofdm_counters *)d_cnt));
        CHECK(ofdm_memcpy_d2h(ctx, totals, d_cnt, sizeof(ofdm_counters) * (size_t)n_snr));
        CHECK(ofdm_ctx_sync(ctx));
        report_rate(!reference_channel ? "channel sweep" : n_taps > 0 ? "multipath sweep" : "sweep", 1, frames, n_sym, n_snr, now_s() - t0);
        ofdm_dev_free(ctx, d_cnt);
    } else {
        uint8_t *bits = NULL;
        CHECK(encode_message(message, &bits, &n_sym));
        const int n_bits = 96 * n_sym, n_words = 3 * n_sym, len = OFDM_FRAME_LEN(n_sym);
        uint32_t *words = (uint32_t *)malloc((size_t)n_words * sizeof(uint32_t));
        uint32_t *rx_words = (uint32_t *)malloc((size_t)n_words * sizeof(uint32_t));
        char *text = (char *)malloc((size_t)n_bits / 8 + 1);
        if (!words || !rx_words || !text) return 1;
        pack_bits(bits, n_bits, words);
        void *d_bits = NULL, *d_frame = NULL, *d_power = NULL, *d_cnt = NULL, *d_rx = NULL;
        CHECK(ofdm_dev_alloc(ctx, &d_bits, (size_t)n_words * 4));
        CHECK(ofdm_dev_alloc(ctx, &d_rx, (size_t)n_words * 4));
        CHECK(ofdm_dev_alloc(ctx, &d_frame, (size_t)len * 8));
        CHECK(ofdm_dev_alloc(ctx, &d_power, 4));
        CHECK(ofdm_dev_alloc(ctx, &d_cnt, sizeof(ofdm_counters)));
        CHECK(ofdm_memcpy_h2d(ctx, d_bits, words, (size_t)n_words * 4));
        CHECK(ofdm_tx_frames(ctx, (const uint32_t *)d_bits, (float *)d_frame, (float *)d_power, 1, n_sym, mode));   /* Transmitter() once, :1191 */
        if (dump) {
            float *iq = (float *)malloc((size_t)len * 8);
            char path[1024];
            CHECK(ofdm_memcpy_d2h(ctx, iq, d_frame, (size_t)len * 8));
            CHECK(ofdm_ctx_sync(ctx));
            snprintf(path, sizeof path, "%s_real.txt", dump);     CHECK(ofdm_write_complex_array_to_file(iq, len, path, 0));
            snprintf(path, sizeof path, "%s_complex.txt", dump);  CHECK(ofdm_write_complex_array_to_file(iq, len, path, 1));
            free(iq);
        }
        /* whole over-the-air path: Transmitter() :569-617 once */
        const int len480 = 160 + len, len_shaped = 2 * len480 + 20, len_rep = 10 * len_shaped;
        const int len_cap = (int)(len_rep * 0.307);                                   /* :945 */
        void *d_f480 = NULL, *d_shaped = NULL, *d_rep = NULL, *d_ota = NULL, *d_cap = NULL, *d_corr = NULL, *d_idx = NULL,
             *d_rxf = NULL, *d_c1 = NULL, *d_c2 = NULL, *d_ld = NULL;
        if (full_chain) {
            CHECK(ofdm_dev_alloc(ctx, &d_f480, (size_t)len480 * 8));   CHECK(ofdm_dev_alloc(ctx, &d_shaped, (size_t)len_shaped * 8));
            CHECK(ofdm_dev_alloc(ctx, &d_rep, (size_t)len_rep * 8));   CHECK(ofdm_dev_alloc(ctx, &d_ota, (size_t)len_rep * 8));
            CHECK(ofdm_dev_alloc(ctx, &d_cap, (size_t)len_cap * 8));   CHECK(ofdm_dev_alloc(ctx, &d_corr, (size_t)len_cap * 4));
            CHECK(ofdm_dev_alloc(ctx, &d_idx, 4));                     CHECK(ofdm_dev_alloc(ctx, &d_rxf, (size_t)len480 * 8));
            CHECK(ofdm_dev_alloc(ctx, &d_c1, (size_t)len480 * 8));     CHECK(ofdm_dev_alloc(ctx, &d_c2, (size_t)len480 * 8));
            CHECK(ofdm_dev_alloc(ctx, &d_ld, (size_t)len * 8));
            CHECK(ofdm_prepend_sts(ctx, (const float *)d_frame, (float *)d_f480, 1, len));                    /* :572-581 */
            CHECK(ofdm_rrc_tx(ctx, (const float *)d_f480, (float *)d_shaped, 1, len480));                     /* :587-605 */
            CHECK(ofdm_gather(ctx, (const float *)d_shaped, NULL, 0, (float *)d_rep, 1, len_shaped, len_rep)); /* :607-612 */
            srand(seed);
        }
        for (int i = 0; i < n_snr; ++i) {                  /* SNR loop :1202-1222 */
            ofdm_rx_dump d;
            memset(&d, 0, sizeof d);
            d.bits = (uint32_t *)d_rx;
            CHECK(ofdm_memset_dev(ctx, d_cnt, 0, sizeof(ofdm_counters)));
            if (full_chain) {
                const int rx_start = rand() % (len_rep - len_cap);                                            /* :949 */
                CHECK(ofdm_awgn_philox_len(ctx, (const float *)d_rep, NULL, SNR[i], seed, (uint32_t)i, 0, (float *)d_ota, 1, len_rep, mode));  /* :1208 */
                CHECK(ofdm_gather(ctx, (const float *)d_ota, NULL, rx_start, (float *)d_cap, 1, len_rep, len_cap));                             /* :955 */
                CHECK(ofdm_packet_detect(ctx, (const float *)d_cap, (float *)d_corr, 1, len_cap));            /* :972 */
                CHECK(ofdm_packet_select(ctx, (const float *)d_corr, (int32_t *)d_idx, 1, len_cap - 47));     /* :978 */
                CHECK(ofdm_rrc_rx_idx(ctx, (const float *)d_cap, (const int32_t *)d_idx, (float *)d_rxf, 1, len_cap, len480));  /* :965, :986-996 */
                CHECK(ofdm_cfo_coarse(ctx, (const float *)d_rxf, (float *)d_c1, NULL, 1, len480));            /* :1004 */
                CHECK(ofdm_cfo_fine(ctx, (const float *)d_c1, (float *)d_c2, NULL, 1, len480));               /* :1012 */
                CHECK(ofdm_gather(ctx, (const float *)d_c2, NULL, 160, (float *)d_ld, 1, len480, len));
                CHECK(ofdm_rx_frames(ctx, (const float *)d_ld, (const uint32_t *)d_bits, 1, n_sym, mode, (ofdm_counters *)d_cnt, &d));  /* :1018-1165 */
            } else
            CHECK(ofdm_awgn_rx_philox(ctx, (const float *)d_frame, (const float *)d_power, (const uint32_t *)d_bits, SNR[i], seed,
                                      (uint32_t)i, 0, 1, n_sym, mode, (ofdm_counters *)d_cnt, &d));
            CHECK(ofdm_memcpy_d2h(ctx, &totals[i], d_cnt, sizeof(ofdm_counters)));
            CHECK(ofdm_memcpy_d2h(ctx, rx_words, d_rx, (size_t)n_words * 4));
            CHECK(ofdm_ctx_sync(ctx));
            if (!quiet) {
                decode_message(rx_words, n_bits, text);
                printf("\n\nFor SNR = %lf \n\nReceived Message: \n%s\n", SNR[i], text);      /* :1204, :1177-1182 */
            }
        }
        if (full_chain) {
            void *all[] = {d_f480, d_shaped, d_rep, d_ota, d_cap, d_corr, d_idx, d_rxf, d_c1, d_c2, d_ld};
            for (unsigned k = 0; k < sizeof all / sizeof all[0]; ++k) ofdm_dev_free(ctx, all[k]);
        }
        ofdm_dev_free(ctx, d_bits); ofdm_dev_free(ctx, d_rx); ofdm_dev_free(ctx, d_frame);
        ofdm_dev_free(ctx, d_power); ofdm_dev_free(ctx, d_cnt);
        free(bits); free(words); free(rx_words); free(text);
    }

    for (int i = 0; i < n_snr; ++i) {
        float Res[3];                                      /* EVM_dB, EVM_AGC_DB, BER  :1210 */
        CHECK(ofdm_counters_finalize(&totals[i], Res));
        EVM_dB[i] = Res[0]; EVM_AGC_dB[i] = Res[1]; BER[i] = Res[2];
        if (!quiet) printf("\nSNR %5.1f dB  EVM dB = %lf  EVM_AGC dB = %lf  BER = %le  (%llu frames)", SNR[i], Res[0], Res[1], Res[2],
                           (unsigned long long)totals[i].frames);
    }
    char path[1024];
    snprintf(path, sizeof path, "%s/Output_SNR.txt", outdir);         CHECK(ofdm_write_float_array_to_file(SNR, n_snr, path));
    snprintf(path, sizeof path, "%s/Output_EVM_AGC.txt", outdir);     CHECK(ofdm_write_float_array_to_file(EVM_dB, n_snr, path));
    snprintf(path, sizeof path, "%s/Output_EVM_AGC_DB.txt", outdir);  CHECK(ofdm_write_float_array_to_file(EVM_AGC_dB, n_snr, path));
    snprintf(path, sizeof path, "%s/Output_BER.txt", outdir);         CHECK(ofdm_write_float_array_to_file(BER, n_snr, path));
    if (!quiet) printf("\nCode Run Successful!\n");
    if (ctx) ofdm_ctx_destroy(ctx);
    return 0;
}
