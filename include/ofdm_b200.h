/*
 * ofdm_b200.h -- C-ABI of libofdm_b200.so: the B200-native (sm_100a) 802.11a OFDM QPSK
 * TX -> AWGN -> RX stage chain.  Plain pointers and sizes only; no torch / C++ types.
 *
 * The reference (Unalome81/IEEE-802.11-OFDM-QPSK-Simulator) has no FFI: its "stage interface"
 * is the set of C functions in src/OFDM.c called from main().  Each entry point below is the
 * batched, re-entrant replacement of one of those functions or inline blocks (cited as
 * OFDM.c:line), plus fused entry points that run several stages in one kernel.  Differences
 * that are deliberate and uniform:
 *   - an explicit context handle instead of the reference's globals (OFDM.c:24-34);
 *   - int status returns instead of exit(1)/perror (OFDM.c:150-153, :97-100);
 *   - caller-owned flat buffers [frames][samples] instead of callee-allocated row pointers;
 *   - IQ is interleaved (re, im) float pairs == the memory layout of C `float complex`;
 *   - payload bits are packed, 96 bits per OFDM symbol = 3 little-endian uint32 words
 *     (bit j of a symbol = bit (j & 31) of word j >> 5); ofdm_pack_bits/ofdm_unpack_bits convert
 *     from/to the one-value-per-bit layout the reference uses (it stores bits as float complex);
 *   - frame = LTS(160 samples) || n_sym x (16-sample CP + 64): the reference's 480-sample frame
 *     (OFDM.c:569-581) minus the 160-sample STS slot, which only detection/coarse CFO use.
 *
 * Pointers documented "device" are CUDA device pointers (from ofdm_dev_alloc or any CUDA
 * allocator, e.g. a torch tensor's data_ptr); "host" pointers are ordinary memory.  All device
 * work is enqueued on the context's stream; entry points that return results to host memory
 * synchronise that stream before returning.  There is no CPU fallback anywhere.  An ofdm_ctx is bound to one GPU and is
 * not thread-safe: use one context per host thread (or per GPU, as host/ofdm_main.c does for its multi-GPU sweep).
 *
 * mode: OFDM_MODE_EXACT reproduces the reference's arithmetic bit for bit (double twiddle
 * products rounded to float, float add/sub, double-widened complex division; SURVEY.md
 * section 7); OFDM_MODE_FAST is the fp32 radix-8 path (1e-5 relative on IQ / EVM).
 */
#ifndef OFDM_B200_H
#define OFDM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OFDM_B200_VERSION 100

enum {
    OFDM_OK = 0,
    OFDM_ERR_INVALID = 1,    /* bad argument (null pointer, n_sym < 1, unknown mode ...) */
    OFDM_ERR_CUDA = 2,       /* a CUDA runtime call failed; see ofdm_last_error() */
    OFDM_ERR_NOMEM = 3,      /* host or device allocation failed (reference: exit(1), OFDM.c:152) */
    OFDM_ERR_IO = 4,         /* fopen/fwrite failed (reference: perror + return, OFDM.c:97-100) */
    OFDM_ERR_NODEVICE = 5    /* no CUDA device: there is NO CPU fallback */
};

enum { OFDM_MODE_EXACT = 0, OFDM_MODE_FAST = 1 };

#define OFDM_NFFT 64
#define OFDM_CP 16
#define OFDM_SYM_LEN 80          /* CP + NFFT */
#define OFDM_LTS_LEN 160
#define OFDM_DATA_PER_SYM 48
#define OFDM_BITS_PER_SYM 96
#define OFDM_WORDS_PER_SYM 3
#define OFDM_MAX_SYM 512
#define OFDM_FRAME_LEN(n_sym) (OFDM_LTS_LEN + OFDM_SYM_LEN * (n_sym))

typedef struct ofdm_ctx ofdm_ctx;

/* Cross-frame totals for one SNR point.  The reference's Res[3] (OFDM.c:1163-1165) is defined
 * per frame with float accumulators that stall at 2^24 (SURVEY.md Q11); batches use integer
 * and double totals and ofdm_counters_finalize() turns them back into {EVM_dB, EVM_AGC_dB, BER}. */
typedef struct {
    uint64_t bit_errors;        /* sum |tx_bit - rx_bit|                         OFDM.c:1156-1159 */
    uint64_t bits;              /* 96 * n_sym * frames                                            */
    uint64_t frames_in_error;   /* frames with >= 1 bit error                                     */
    uint64_t rail_errors;       /* I/Q rails whose slicer output != tx rail      OFDM.c:1134-1142 */
    uint64_t frames;
    double sum_err2;            /* sum |equalised - tx|^2 over data bins         OFDM.c:1114-1115 */
    double sum_ref2;            /* sum |tx|^2 over data bins                     OFDM.c:1116      */
    double sum_evm_lin;         /* sum over frames of the per-frame linear EVM   OFDM.c:1124      */
} ofdm_counters;

/* Optional per-frame / per-bin outputs of the receiver (device pointers, any may be NULL). */
typedef struct {
    float *H;                   /* [frames][64][2]        channel estimate, centred order  OFDM.c:848        */
    float *eq;                  /* [frames][n_sym*48][2]  equalised data bins              OFDM.c:1050,:1063 */
    float *sliced;              /* [frames][n_sym*48][2]  "AGC" slicer output              OFDM.c:852        */
    uint32_t *bits;             /* [frames][n_sym*3]      demodulated bits, packed         OFDM.c:873        */
    int32_t *frame_bit_errors;  /* [frames]                                                                  */
    float *frame_evm_lin;       /* [frames]               per-frame EVM before the slicer  OFDM.c:1124       */
} ofdm_rx_dump;

/* ---- context, errors, memory ---------------------------------------------------------------- */
int ofdm_version(void);
const char *ofdm_strerror(int status);
int ofdm_ctx_create(ofdm_ctx **ctx, int device);
int ofdm_ctx_destroy(ofdm_ctx *ctx);
const char *ofdm_last_error(const ofdm_ctx *ctx);
int ofdm_ctx_set_stream(ofdm_ctx *ctx, void *cuda_stream);   /* run on a caller-owned cudaStream_t */
void *ofdm_ctx_stream(const ofdm_ctx *ctx);
int ofdm_ctx_sync(ofdm_ctx *ctx);
/* tuning / testing knobs:
 *   "force_generic_rx"  = 1  routes every receiver call through the generic kernel
 *   "exact_speculation" = 0  OFDM_MODE_EXACT sweeps run the reference's arithmetic on every frame instead of
 *                            speculating in fp32, verifying, and replaying doubtful frames exactly (default 1;
 *                            both give the same error counts, DESIGN.md section 4)
 *   "force_replay"      = 1  the verification fails on every frame (exercises the replay path)
 *   "stream_layout"     = 1  the fused receivers and the fused Monte-Carlo sweep give a warp one frame at a time (k_stream_rx2 /
 *                            k_stream_rxn / k_mc_philox) instead of one frame per 8-lane group (k_stream_quad / k_mc_quad,
 *                            default 0; same totals in EXACT mode, DESIGN.md sections 4.5, 4.6)
 *   "stream_warps"      = 8  k_stream_quad in blocks of 8 warps (128 registers) instead of 6 (168 registers, default)
 *   "general_stream"    = 1  two-symbol frames take the build that serves every other frame shape too (k_stream_quad without its
 *                            compile-time ring slots; with "stream_layout" = 1: the multi-pass k_stream_rxn)
 *   "evm_guard"         = N  bins whose channel estimate is smaller than N error radii are replayed exactly (default 820): the
 *                            EVM sums' distance from the all-exact kernel's against the number of replays (DESIGN.md section 4)
 *   "power_margin"      = N  the exact frame power speculates each term of the serial float sum as x^2 + y^2 and takes the
 *                            reference's hypot()^2 where the running sum is within N double ulps of a tie between two floats
 *                            (default 16, the proven bound is 7; 2^28 = the reference's operations on every sample; same floats)
 *   "fused_sweep"       = 0  injected-noise sweeps launch one channel+receiver kernel per SNR point instead of the all-SNR
 *                            kernel (default 1; same totals)
 *   "multipath_path"    = 0  Monte-Carlo sweeps of the reference channel with taps (ofdm_mc_sweep_multipath_dev and the
 *                            other sweeps given taps) pick the faster of their two implementations per mode (default);
 *                       = 1  frames staged in HBM (TX, fading, power, one receiver kernel per SNR point);
 *                       = 2  the fused on-chip kernel; both give the same totals */
int ofdm_ctx_set_option(ofdm_ctx *ctx, const char *name, int value);
/* frames (sweeps: frame x SNR points) the speculating kernels of THIS context replayed in the reference's arithmetic since
 * its creation / the last reset */
int ofdm_ctx_replayed_frames(ofdm_ctx *ctx, uint64_t *count, int reset);
int ofdm_ctx_sm_count(const ofdm_ctx *ctx);
uint64_t ofdm_ctx_launch_count(const ofdm_ctx *ctx);          /* kernels launched so far by this ctx */
int ofdm_dev_alloc(ofdm_ctx *ctx, void **ptr, size_t bytes);
int ofdm_dev_free(ofdm_ctx *ctx, void *ptr);
int ofdm_host_alloc(ofdm_ctx *ctx, void **ptr, size_t bytes);   /* pinned host memory */
int ofdm_host_free(ofdm_ctx *ctx, void *ptr);
int ofdm_memcpy_h2d(ofdm_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);   /* async on the stream */
int ofdm_memcpy_d2h(ofdm_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);   /* async on the stream */
int ofdm_memset_dev(ofdm_ctx *ctx, void *dst_dev, int value, size_t bytes);

/* ---- stage-level entry points (device buffers) ---------------------------------------------- */
/* layout helpers: one byte per bit <-> packed words */
int ofdm_pack_bits(ofdm_ctx *ctx, const uint8_t *bits_dev, uint32_t *packed_dev, long n_symbols);
int ofdm_unpack_bits(ofdm_ctx *ctx, const uint32_t *packed_dev, uint8_t *bits_dev, long n_symbols);
/* QPSK_Modulator, OFDM.c:415-433: n_symbols x 96 bits -> [n_symbols][48] points */
int ofdm_qpsk_modulate(ofdm_ctx *ctx, const uint32_t *bits_dev, float *mod_dev, long n_symbols);
/* inline frame build, OFDM.c:523-548: [n_symbols][48] -> centred [n_symbols][64] grid, pilots +1,+1,+1,-1 */
int ofdm_map_subcarriers(ofdm_ctx *ctx, const float *mod_dev, float *grid_dev, long n_symbols);
/* ifft, OFDM.c:320-339: centred input, output rotated by 32 samples exactly as the reference's (SURVEY Q4) */
int ofdm_ifft64(ofdm_ctx *ctx, const float *in_dev, float *out_dev, long n, int mode);
/* fft, OFDM.c:314-318: centred (fft_shift'ed) output */
int ofdm_fft64(ofdm_ctx *ctx, const float *in_dev, float *out_dev, long n, int mode);
/* CP add, OFDM.c:559-565: [n][64] -> [n][80] */
int ofdm_add_cp(ofdm_ctx *ctx, const float *sym_dev, float *out_dev, long n);
/* Preamble_Generator(type=1), OFDM.c:368-399: host copies of the LTS, frequency (centred, 64) and time (160) */
int ofdm_lts(ofdm_ctx *ctx, float *lts_freq_host, float *lts_time_host);
/* Transmitter OFDM.c:500-581 without STS/RRC: bits -> frames [n_frames][160+80*n_sym]; power_dev
 * (nullable, [n_frames]) receives the per-frame mean power of OFDM.c:637-643 */
int ofdm_tx_frames(ofdm_ctx *ctx, const uint32_t *bits_dev, float *frames_dev, float *power_dev,
                   long n_frames, int n_sym, int mode);
/* signal-power block of Transmission_Over_Air, OFDM.c:637-643 (float accumulator, sequential, in EXACT) */
int ofdm_frame_power(ofdm_ctx *ctx, const float *frames_dev, float *power_dev, long n_frames, int frame_len, int mode);
/* Transmission_Over_Air, OFDM.c:635-655, real-rail noise only (SURVEY Q1-Q3), per-frame power.
 * _inject: the standard-normal draw per sample is supplied (g_dev [n_frames][frame_len]);
 * _philox: drawn on chip, key (seed, stream), counter (frame0 + frame, block, domain).
 * power_dev may be NULL (computed internally). */
int ofdm_awgn_inject(ofdm_ctx *ctx, const float *tx_dev, const float *g_dev, const float *power_dev, float snr_db,
                     float *ota_dev, long n_frames, int n_sym, int mode);
int ofdm_awgn_philox(ofdm_ctx *ctx, const float *tx_dev, const float *power_dev, float snr_db, uint32_t seed,
                     uint32_t stream, uint64_t frame0, float *ota_dev, long n_frames, int n_sym, int mode);

/* ---- channels (no reference counterpart: the reference's channel is OFDM_NOISE_REAL_RAIL + OFDM_SNR_FRAME_POWER) ----
 * noise:   OFDM_NOISE_REAL_RAIL  all of the noise power np on the I rail, y.re = x.re + sqrt(np) g0, y.im = x.im (SURVEY Q1);
 *          OFDM_NOISE_COMPLEX    circular complex noise of total variance np, y = x + sqrt(np/2) (g0 + i g1).
 * snr_def: OFDM_SNR_FRAME_POWER  np = P / (float)pow(10, snr_db/10), P the per-frame power of OFDM.c:637-643 (after the taps);
 *          OFDM_SNR_ESN0         Es/N0 per data subcarrier: np = (float)(1 / (64 * 10^(snr_db/10))), the same for every frame;
 *          OFDM_SNR_EBN0         Eb/N0, 2 bits per QPSK point: np = (float)(1 / (128 * 10^(snr_db/10))).
 * n_taps:  0 = AWGN, 1..16 = the multipath channel of configs[4] below in front of the noise.
 * g0 is the Philox domain-0 normal the real-rail channel draws for the sample, g1 the normal in the same slot of domain 4.
 * EXACT: sigma_d = sqrt((double)np) (real rail) or sqrt(0.5 * (double)np) (complex), each noisy rail x + (float)(sigma_d * g);
 * FAST: fmaf(sigma_f, g, x).  {OFDM_NOISE_REAL_RAIL, OFDM_SNR_FRAME_POWER, n} is the reference's channel and runs exactly the
 * code of ofdm_awgn_philox / ofdm_mc_sweep_points_dev / ofdm_mc_sweep_until. */
enum { OFDM_NOISE_REAL_RAIL = 0, OFDM_NOISE_COMPLEX = 1 };
enum { OFDM_SNR_FRAME_POWER = 0, OFDM_SNR_ESN0 = 1, OFDM_SNR_EBN0 = 2 };
typedef struct { int noise, snr_def, n_taps; } ofdm_channel;
/* the channel on LTS||data frames, Philox draws as ofdm_awgn_philox; power_dev (nullable) is computed when snr_def needs it and
 * ignored otherwise.  Chained with ofdm_rx_frames it gives per-bin dumps (e.g. constellations) under any channel. */
int ofdm_awgn_philox_ex(ofdm_ctx *ctx, int noise, int snr_def, const float *tx_dev, const float *power_dev, float snr_db,
                        uint32_t seed, uint32_t stream, uint64_t frame0, float *ota_dev, long n_frames, int n_sym, int mode);
/* Receiver OFDM.c:1018-1165 on LTS||data frames: Channel_Estimation :830, CP strip :1024, fft :1037,
 * equalise :1046, demap :1061, AGC_Receiver :852, QPSK_Demodulator :873, EVM :1106-1150, BER :1154.
 * counters_dev (device, one ofdm_counters, accumulated into -- zero it first) may be NULL. */
int ofdm_rx_frames(ofdm_ctx *ctx, const float *ota_dev, const uint32_t *tx_bits_dev, long n_frames, int n_sym,
                   int mode, ofdm_counters *counters_dev, const ofdm_rx_dump *dump);
/* fused channel + receiver: reads TX frames, adds the noise in registers, never writes OTA IQ */
int ofdm_awgn_rx_inject(ofdm_ctx *ctx, const float *tx_dev, const float *g_dev, const float *power_dev,
                        const uint32_t *tx_bits_dev, float snr_db, long n_frames, int n_sym, int mode,
                        ofdm_counters *counters_dev, const ofdm_rx_dump *dump);
int ofdm_awgn_rx_philox(ofdm_ctx *ctx, const float *tx_dev, const float *power_dev, const uint32_t *tx_bits_dev,
                        float snr_db, uint32_t seed, uint32_t stream, uint64_t frame0, long n_frames, int n_sym,
                        int mode, ofdm_counters *counters_dev, const ofdm_rx_dump *dump);

/* the same over a list of SNR points (device buffers, counters_dev [n_snr] accumulated into, no synchronisation): for
 * two-symbol frames this is ONE kernel for the whole list (k_sweep_lin: the transform is linear, so each frame and its
 * draws are transformed once and every SNR point costs a multiply-add per bin plus the decision stage; EXACT mode keeps
 * the reference's error counts by verification + exact replay, DESIGN.md section 4); other shapes launch per point. */
int ofdm_awgn_rx_inject_sweep(ofdm_ctx *ctx, const float *tx_dev, const float *g_dev, const float *power_dev,
                              const uint32_t *tx_bits_dev, const float *snr_db, int n_snr, long n_frames, int n_sym, int mode,
                              ofdm_counters *counters_dev);

/* ---- the receiver's stages one by one (device buffers; what ofdm_rx_frames fuses) ------------------------------------
 * 1:1 batched counterparts of the reference's receiver functions and inline blocks, so that a caller can stop after any
 * stage exactly as with the reference.  Chained -- strip_cp, fft64, channel_estimate, equalize, demap, agc_slicer,
 * qpsk_demodulate -- they reproduce the reference's H_est, equalised points, slicer output and bits bit for bit in EXACT mode.
 * ofdm_strip_cp         CP strip, OFDM.c:1024-1031: frames [n][frame_len] -> bodies [n][n_sym][64]; data_off = index of the
 *                       first data symbol's CP (160 for LTS || data frames, 320 for the reference's STS || LTS || data frame)
 * ofdm_channel_estimate Channel_Estimation, OFDM.c:830-850: H [n][64] centred = 0.5 (fft(LTS half 1) + fft(LTS half 2)) conj(L);
 *                       lts_off = index of the LTS slot (0, or 160 behind an STS slot: the reference reads samples 192..319)
 * ofdm_equalize         one-tap ZF, OFDM.c:1044-1052: E [n][n_sym][64] = F / H on all 64 bins (libgcc __divsc3 in EXACT mode;
 *                       the 12 null bins hold the inf / NaN the reference computes there and never reads)
 * ofdm_demap            OFDM.c:1059-1069: [n_symbols][64] -> the 48 data bins [n_symbols][48]
 * ofdm_agc_slicer       AGC_Receiver, OFDM.c:852-871: each rail -> +1/sqrt(2) if > 0 else -1/sqrt(2)
 * ofdm_qpsk_demodulate  QPSK_Demodulator, OFDM.c:873-908: [n_symbols][48] points -> packed bits [n_symbols][3] */
int ofdm_strip_cp(ofdm_ctx *ctx, const float *frames_dev, float *bodies_dev, long n_frames, int n_sym, int frame_len, int data_off);
int ofdm_channel_estimate(ofdm_ctx *ctx, const float *frames_dev, float *H_dev, long n_frames, int frame_len, int lts_off, int mode);
int ofdm_equalize(ofdm_ctx *ctx, const float *F_dev, const float *H_dev, float *E_dev, long n_frames, int n_sym, int mode);
int ofdm_demap(ofdm_ctx *ctx, const float *grid_dev, float *points_dev, long n_symbols);
int ofdm_agc_slicer(ofdm_ctx *ctx, const float *points_dev, float *sliced_dev, long n_symbols);
int ofdm_qpsk_demodulate(ofdm_ctx *ctx, const float *points_dev, uint32_t *bits_dev, long n_symbols);

/* ---- sweep drivers: host buffers in, host counters out (what main()'s loop OFDM.c:1202-1222 does) ---- */
/* Transmitter once, then per SNR point channel + receiver, injected normals reused across points
 * (only the scale changes).  bits_host [n_frames][n_sym*3] packed; g_host [n_frames][frame_len];
 * out_host [n_snr].  H2D copies, kernels and the D2H of the counters all run inside the call. */
int ofdm_sweep_inject_host(ofdm_ctx *ctx, const uint32_t *bits_host, const float *g_host, long n_frames, int n_sym,
                           const float *snr_db, int n_snr, int mode, ofdm_counters *out_host);
/* same with resident device buffers (no copies except the counters) */
int ofdm_sweep_inject_dev(ofdm_ctx *ctx, const uint32_t *bits_dev, const float *g_dev, long n_frames, int n_sym,
                          const float *snr_db, int n_snr, int mode, ofdm_counters *out_host);

/* ---- on-chip Monte-Carlo (no reference counterpart: the reference draws from libc rand(), OFDM.c:626) ----
 * Counter-based streams, Philox4x32-10: key (seed, stream), counter (frame_lo, frame_hi, block, domain);
 * payload bits: domain 1, block = symbol index, words 0..2; noise: domain 0, stream = index of the SNR point,
 * block layout in DESIGN.md.  Results depend only on (seed, frame0 + frame index), never on the GPU count. */
int ofdm_random_bits(ofdm_ctx *ctx, uint32_t seed, uint64_t frame0, long n_frames, int n_sym, uint32_t *bits_dev);
/* Whole sweep fused in one kernel for n_sym == 2 (bits, TX, channel, RX, counters; nothing else touches HBM);
 * other n_sym run the same streams through the staged kernels.  n_snr <= 64.  _dev accumulates into device
 * counters [n_snr] without synchronising (for a following NCCL all-reduce); the other returns host totals. */
int ofdm_mc_sweep_philox_dev(ofdm_ctx *ctx, uint32_t seed, uint64_t frame0, long n_frames, int n_sym,
                             const float *snr_db, int n_snr, int mode, ofdm_counters *counters_dev);
int ofdm_mc_sweep_philox(ofdm_ctx *ctx, uint32_t seed, uint64_t frame0, long n_frames, int n_sym,
                         const float *snr_db, int n_snr, int mode, ofdm_counters *out_host);

/* The same over an explicit list of points: streams[i] (NULL: i) is the Philox noise stream of point i, so that a caller
 * can drop finished SNR points from the list without changing the draws of the others; n_taps = 0 is the AWGN channel,
 * 1..16 the multipath channel of configs[4] below.  n_points <= 64.  Accumulates into counters_dev, no synchronisation. */
int ofdm_mc_sweep_points_dev(ofdm_ctx *ctx, uint32_t seed, uint64_t frame0, long n_frames, int n_sym, int n_taps,
                             const float *snr_db, const uint32_t *streams, int n_points, int mode, ofdm_counters *counters_dev);
/* configs[3] as BASELINE.json states it: every SNR point runs until it has >= target_errors bit errors or >= max_bits
 * bits (the BER budget: 100 errors / 1e-7 = 1e9 bits), whichever comes first.  Frames are consumed in rounds of round_frames
 * (global frame indices frame0 + r * round_frames ...); after a round the finished points leave the kernel's list.  The
 * stop decisions are taken at round boundaries on totals, so the result depends only on (seed, frame0, round_frames): a
 * multi-GPU driver that splits each round's frame range across ranks and all-reduces the round's counters before
 * deciding reproduces it exactly (host/ofdm_main.c --target-errors; sweep.mc_sweep_until).  out_host [n_snr]; rounds_out nullable. */
int ofdm_mc_sweep_until(ofdm_ctx *ctx, uint32_t seed, uint64_t frame0, int n_sym, int n_taps, const float *snr_db, int n_snr,
                        int mode, uint64_t target_errors, uint64_t max_bits, long round_frames, ofdm_counters *out_host,
                        int *rounds_out);
/* The two above through any channel (ofdm_channel, see ofdm_awgn_philox_ex); ofdm_mc_sweep_points_dev and ofdm_mc_sweep_until are
 * these with {OFDM_NOISE_REAL_RAIL, OFDM_SNR_FRAME_POWER, n_taps}.  Other channels run FAST two-symbol sweeps fused on chip
 * (k_mc_quad) and everything else -- all of EXACT -- staged: Philox bits, transmitter, [taps], [frame power], then per point
 * the channel into HBM and the verified receiver of ofdm_rx_frames.  Results depend only on (seed, global frame index, stream).
 * A NULL or invalid channel returns OFDM_ERR_INVALID. */
int ofdm_mc_sweep_channel_dev(ofdm_ctx *ctx, const ofdm_channel *ch, uint32_t seed, uint64_t frame0, long n_frames, int n_sym,
                              const float *snr_db, const uint32_t *streams, int n_points, int mode, ofdm_counters *counters_dev);
int ofdm_mc_sweep_channel_until(ofdm_ctx *ctx, const ofdm_channel *ch, uint32_t seed, uint64_t frame0, int n_sym, const float *snr_db,
                                int n_snr, int mode, uint64_t target_errors, uint64_t max_bits, long round_frames,
                                ofdm_counters *out_host, int *rounds_out);

/* ---- the coded link: the 802.11a convolutional code (IEEE 802.11a section 17.3.5.6; definitions in DESIGN.md section 6.2) ----
 * K = 7, g0 = 133 (octal, output A), g1 = 171 (output B), rate 1/2 (48 data bits per OFDM symbol) or 3/4 (72: A0 B0 A1 B2 of every
 * three input bits), per-symbol interleaver i = 6 (k mod 16) + floor(k / 16), and a precoding onto this project's QPSK map that sends
 * coded bit c0 on the I rail and c1 on the Q rail as the 802.11a constellation (2c - 1)/sqrt(2).  A frame of n_sym symbols carries
 * K_info = n_sym N_DBPS - 6 information bits -- bits 0 .. K_info-1 of its packed words -- and 6 zero tail bits.
 * ofdm_conv_encode     information words [n_frames][n_sym*3] -> payload words [n_frames][n_sym*3] for ofdm_tx_frames.
 * ofdm_viterbi_decode  maximum-likelihood decoding of whole frames from the receiver's H [n_frames][64][2] and eq
 *                      [n_frames][n_sym*48][2] dumps: soft (L = |H|^2 eq per rail) or hard (L = +-1 by the slicer's rule) decisions.
 *                      decoded_dev [n_frames][n_sym*3] (nullable) receives the decoded information bits (tail and pad bits 0);
 *                      counters_dev (nullable; needs info_dev) accumulates the coded counters.
 * Coded counters: bit_errors = information-bit errors, bits = K_info x frames, frames_in_error = packets with >= 1 such error
 * (PER = frames_in_error / frames), rail_errors and the three sums 0.  Raw counters: the receiver's own against the payload words
 * (rail_errors = coded-bit errors; the EVM sums keep their meaning).
 * ofdm_mc_sweep_coded_dev / _until: ofdm_mc_sweep_channel_dev / _until with the code between the Philox bits and the transmitter
 * and the decoder behind the receiver, always staged through HBM; an Eb/N0 point counts information bits (Es/N0 = Eb/N0 x 2R).
 * raw (nullable) receives the raw counters; the until rule stops on the coded ones.  A NULL or invalid code or channel returns
 * OFDM_ERR_INVALID. */
enum { OFDM_CODE_R12 = 1, OFDM_CODE_R34 = 2 };
enum { OFDM_DECISION_SOFT = 0, OFDM_DECISION_HARD = 1 };
typedef struct { int rate, decision; } ofdm_code;
int ofdm_conv_encode(ofdm_ctx *ctx, int rate, const uint32_t *info_dev, uint32_t *payload_dev, long n_frames, int n_sym);
int ofdm_viterbi_decode(ofdm_ctx *ctx, const ofdm_code *code, const float *H_dev, const float *eq_dev,
                        const uint32_t *info_dev /* nullable: count against it */, uint32_t *decoded_dev /* nullable */,
                        long n_frames, int n_sym, ofdm_counters *counters_dev /* nullable */);
int ofdm_mc_sweep_coded_dev(ofdm_ctx *ctx, const ofdm_channel *ch, const ofdm_code *code, uint32_t seed, uint64_t frame0,
                            long n_frames, int n_sym, const float *snr_db, const uint32_t *streams, int n_points, int mode,
                            ofdm_counters *coded_dev, ofdm_counters *raw_dev /* nullable */);
int ofdm_mc_sweep_coded_until(ofdm_ctx *ctx, const ofdm_channel *ch, const ofdm_code *code, uint32_t seed, uint64_t frame0,
                              int n_sym, const float *snr_db, int n_snr, int mode, uint64_t target_errors, uint64_t max_bits,
                              long round_frames, ofdm_counters *coded_host, ofdm_counters *raw_host /* nullable */, int *rounds_out);

/* ---- multipath extension (BASELINE configs[4]; the reference's only channel is AWGN, OFDM.c:635-655) ----
 * y[n] = sum_l h[l] x[n-l] per frame, n_taps <= 16 (= CP length), applied between the transmitter and
 * Transmission_Over_Air; the reference's own LTS estimate + one-tap equaliser (OFDM.c:830-850, 1046-1052) undo it.
 * _taps: taps supplied, [n_frames][n_taps] complex; _philox: drawn on chip (i.i.d. CN(0, 1/n_taps), Philox
 * domain 2), optionally written to taps_out_dev.  out_dev must differ from tx_dev. */
int ofdm_multipath_taps(ofdm_ctx *ctx, const float *tx_dev, const float *taps_dev, int n_taps, float *out_dev,
                        long n_frames, int n_sym);
int ofdm_multipath_philox(ofdm_ctx *ctx, const float *tx_dev, uint32_t seed, uint64_t frame0, int n_taps,
                          float *out_dev, float *taps_out_dev, long n_frames, int n_sym);
/* Monte-Carlo sweep through the multipath channel (bits, taps and noise from the Philox streams), accumulating
 * into device counters [n_snr]; the signal power of OFDM.c:637-643 is measured after the channel. */
int ofdm_mc_sweep_multipath_dev(ofdm_ctx *ctx, uint32_t seed, uint64_t frame0, long n_frames, int n_sym, int n_taps,
                                const float *snr_db, int n_snr, int mode, ofdm_counters *counters_dev);

/* ---- pulse shaping (SURVEY 8(f) rank 1: the blocks either side of the stage chain on the wire) ----
 * ofdm_rrc_tx: x2 zero-stuff + 21-tap RRC (RRC_Filter_Tx, OFDM.c:32) full convolution, OFDM.c:587-605 with Convolution()
 *   OFDM.c:342-364: [n_frames][frame_len] -> [n_frames][2*frame_len + 20].
 * ofdm_rrc_rx: matched filter + decimation, OFDM.c:959-996: full convolution of in_len samples, then every 2nd sample
 *   from packet_idx, frame_len of them.  packet_idx = 20 re-aligns a frame shaped by ofdm_rrc_tx (the reference finds
 *   it with Packet_Detection/Packet_Selection: ofdm_packet_detect / ofdm_packet_select below, then ofdm_rrc_rx_idx).
 * ofdm_awgn_inject_len: Transmission_Over_Air (OFDM.c:635) on frames of any length, e.g. the oversampled waveform. */
int ofdm_rrc_tx(ofdm_ctx *ctx, const float *frames_dev, float *out_dev, long n_frames, int frame_len);
int ofdm_rrc_rx(ofdm_ctx *ctx, const float *in_dev, float *out_dev, long n_frames, int in_len, int packet_idx, int frame_len);
int ofdm_awgn_inject_len(ofdm_ctx *ctx, const float *tx_dev, const float *g_dev, const float *power_dev, float snr_db,
                         float *ota_dev, long n_frames, int frame_len, int mode);
/* same with on-chip Philox draws (domain 3: sample n of a frame takes normal n & 3 of block n >> 2) */
int ofdm_awgn_philox_len(ofdm_ctx *ctx, const float *tx_dev, const float *power_dev, float snr_db, uint32_t seed, uint32_t stream,
                         uint64_t frame0, float *ota_dev, long n_frames, int frame_len, int mode);

/* ---- packet detection / selection (SURVEY 8(f) rank 2), batched over n captures of len samples ----
 * ofdm_packet_detect: Packet_Detection, OFDM.c:659-683 (delay 16, window 32, no conjugate): corr_dev [n][len-47],
 *   the real part the reference stores in Corr_Out (its imaginary part is always 0).
 * ofdm_packet_select: Packet_Selection, OFDM.c:685-771: idx_dev [n] = packet index (candidate + 11), 0 when detection
 *   fails, as the reference.  The reference reads Corr_Out[candidate+230] without a bound check; lags beyond the
 *   array count as below threshold here. */
int ofdm_packet_detect(ofdm_ctx *ctx, const float *rx_dev, float *corr_dev, long n, int len);
int ofdm_packet_select(ofdm_ctx *ctx, const float *corr_dev, int32_t *idx_dev, long n, int len_corr);

/* ---- CFO stages and full-path glue (SURVEY 8(f) ranks 3, 4) ----
 * Frames here are the reference's 480-sample layout STS(160) || LTS(160) || data (OFDM.c:569-581) or longer.
 * ofdm_sts: host copy of the short-preamble slot, Preamble_Generator(type 0), OFDM.c:479-492 (bit-exact).
 * ofdm_prepend_sts: [n][frame_len] -> [n][160 + frame_len] (OFDM.c:572-581).
 * ofdm_gather: out[f][j] = in[f][(start_f + j) % in_len], j < out_len; start_dev [n] or NULL + start_scalar.  This is
 *   Slice_Repeater (OFDM.c:193): tiling (x10 repetition :607-612: start 0, out_len = 10*in_len), capture windows
 *   (:945-955) and plain slices (dropping the STS: start 160).
 * ofdm_rrc_rx_idx: ofdm_rrc_rx with a per-capture packet index (OFDM.c:978-996); filtered samples past the capture
 *   (an out-of-bounds read in the reference when a packet starts late) count as zero.
 * ofdm_cfo_coarse / ofdm_cfo_fine: Coarse_CFO_Estimation OFDM.c:773-804 (STS slots 5/6) and Fine_CFO_Estimation
 *   OFDM.c:806-828 (LTS halves): estimate + derotation; freq_dev [n] (nullable) receives the float estimates.
 *   The reference calls double libm atan2 / cexp here; agreement is specified to 1e-6 relative (see DESIGN.md). */
int ofdm_sts(ofdm_ctx *ctx, float *sts_time_host);
int ofdm_prepend_sts(ofdm_ctx *ctx, const float *frames_dev, float *out_dev, long n_frames, int frame_len);
int ofdm_gather(ofdm_ctx *ctx, const float *in_dev, const int32_t *start_dev, int start_scalar, float *out_dev, long n,
                int in_len, int out_len);
int ofdm_rrc_rx_idx(ofdm_ctx *ctx, const float *in_dev, const int32_t *idx_dev, float *out_dev, long n_frames, int in_len,
                    int frame_len);
int ofdm_cfo_coarse(ofdm_ctx *ctx, const float *rx_dev, float *out_dev, float *freq_dev, long n, int len);
int ofdm_cfo_fine(ofdm_ctx *ctx, const float *rx_dev, float *out_dev, float *freq_dev, long n, int len);

/* Multi-GPU glue: split device counters [n] into homogeneous buffers (ints [n][5] uint64: bit_errors, bits,
 * frames_in_error, rail_errors, frames; dbls [n][3]: sum_err2, sum_ref2, sum_evm_lin) for a sum all-reduce
 * (ncclUint64 / ncclDouble), and merge them back.  The all-reduce is the path's only exchange (SURVEY 8(e)). */
int ofdm_counters_pack(ofdm_ctx *ctx, const ofdm_counters *counters_dev, int n, uint64_t *ints_dev, double *dbls_dev);
int ofdm_counters_unpack(ofdm_ctx *ctx, ofdm_counters *counters_dev, int n, const uint64_t *ints_dev, const double *dbls_dev);

/* Res[3] = {EVM_dB, EVM_AGC_dB, BER} of OFDM.c:1163-1165 from batch totals */
int ofdm_counters_finalize(const ofdm_counters *c, float res[3]);

/* ---- result / dump writers (host) ------------------------------------------------------------- */
/* write_float_array_to_file, OFDM.c:123-143: one line, tab-separated %.2e */
int ofdm_write_float_array_to_file(const float *a, int n, const char *fname);
/* write_complex_array_to_file, OFDM.c:94-121.  format 0 = what the reference writes today (real parts
 * only, %.15e, tab-separated; compare_double.py reads it); format 1 = the commented-out line :105 with
 * blanks ("re + imi" / "re - imi" triples, the layout compare_complex.py parses).  SURVEY Q12. */
int ofdm_write_complex_array_to_file(const float *a_iq, int n, const char *fname, int format);

#ifdef __cplusplus
}
#endif
#endif
