// ofdm_b200.cu -- context, launch geometry and the extern "C" boundary of libofdm_b200.so.
// Every entry point of include/ofdm_b200.h is defined here (writers live in host/ofdm_io.c).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <set>
#include <type_traits>
#include <utility>

#include "ofdm_chain.cuh"
#include "ofdm_stream.cuh"
#include "ofdm_mc_quad.cuh"
#include "ofdm_sweep.cuh"
#include "ofdm_code.cuh"

using namespace ofdm;

struct ofdm_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    bool owns_stream = false;
    cudaStream_t copy_stream = nullptr;          // H2D pipeline of ofdm_sweep_inject_host
    cudaEvent_t copy_done[2] = {nullptr, nullptr}, call_start = nullptr;
    uint64_t launches = 0;
    bool force_generic = false;      // testing knob: route n_sym == 2 sweeps through the generic kernel too
    bool checked = true;             // EXACT sweeps speculate in fp32, verify, and replay exactly (kArithChecked)
    bool force_replay = false;       // testing knob: the verification fails every frame
    bool general_stream = false;     // testing knob: two-symbol frames through the multi-pass streaming kernel too
    int stream_warps = 6;            // k_stream_quad: warps per block (6: 168 registers, 12 warps per SM; 8: 128 registers, 16 warps per SM)
    int stream_layout = 0;           // streaming receivers: 0 = one frame per lane group (k_stream_quad), 1 = one frame per warp (k_stream_rx2 / rxn)
    bool fused_sweep = true;         // ofdm_sweep_inject_*: the all-SNR kernel k_sweep_lin (default frame shape) instead of one launch per SNR point
    float evm_guard = kEvmGuard;     // tuning knob: bins with |H| below this many error radii are replayed exactly (EVM accuracy vs replays)
    uint32_t power_margin = 16;      // k_frame_power_tiled: samples whose running sum is within this many double ulps of a float tie take the reference's operations
    int multipath_path = 0;          // configs[4]: 0 = auto (fast: fused on-chip kernel, exact: HBM-staged frames), 1 = staged, 2 = fused
    char err[256] = {0};
    float lts_freq[128];
    float lts_time[320];
    float sts_time[320];
    float *sts_dev = nullptr;
    unsigned long long *replayed_dev = nullptr;  // frames / points the speculating kernels replayed exactly (this context)
    float lts_power_prefix = 0.0f;
    // cached scratch (grown on demand, released with the context); slots 7..10 belong to the coded link: payload words, H and
    // eq dumps, k_viterbi's survivors in HBM
    void *scratch[11] = {nullptr};
    size_t scratch_bytes[11] = {0};
};

namespace {

const signed char kLk[53] = {1, 1, -1, -1, 1, 1, -1, 1, -1, 1, 1, 1, 1, 1, 1, -1, -1, 1, 1, -1, 1, -1, 1, 1, 1, 1, 0,
                             1, -1, -1, 1, 1, -1, 1, -1, 1, -1, -1, -1, -1, -1, 1, 1, -1, -1, 1, -1, 1, -1, 1, 1, 1, 1};

int fail(ofdm_ctx *ctx, int status, const char *what, cudaError_t e = cudaSuccess)
{
    if (ctx) {
        if (e != cudaSuccess) snprintf(ctx->err, sizeof ctx->err, "%s: %s", what, cudaGetErrorString(e));
        else snprintf(ctx->err, sizeof ctx->err, "%s", what);
    }
    return status;
}

#define OFDM_CUDA(ctx, call)                                                   \
    do {                                                                       \
        cudaError_t e_ = (call);                                               \
        if (e_ != cudaSuccess) return fail((ctx), OFDM_ERR_CUDA, #call, e_);   \
    } while (0)

#define OFDM_REQUIRE(ctx, cond)                                                          \
    do {                                                                                 \
        if (!(cond)) return fail((ctx), OFDM_ERR_INVALID, "invalid argument: " #cond);   \
    } while (0)

int check_launch(ofdm_ctx *ctx, const char *name)
{
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, OFDM_ERR_CUDA, name, e);
    ctx->launches += 1;
    return OFDM_OK;
}

int bind(ofdm_ctx *ctx)
{
    if (!ctx) return OFDM_ERR_INVALID;
    OFDM_CUDA(ctx, cudaSetDevice(ctx->device));
    return OFDM_OK;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device property of a kernel: set once per (kernel, device), not per launch
template <typename K>
cudaError_t allow_smem(ofdm_ctx *ctx, K kernel, size_t bytes)
{
    static std::mutex mu;
    static std::set<std::pair<const void *, int>> done;
    std::lock_guard<std::mutex> lock(mu);
    const std::pair<const void *, int> key(reinterpret_cast<const void *>(kernel), ctx->device);
    if (done.count(key)) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) done.insert(key);
    return e;
}

// persistent launch geometry: resident blocks per SM (from the occupancy calculator) x SM count,
// capped by the amount of work
template <typename K>
int grid_for(ofdm_ctx *ctx, K kernel, size_t dyn_smem, long work_items_per_block_iter, long work, int threads = kThreads)
{
    int per_sm = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, dyn_smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    long full = (long)per_sm * ctx->sm_count;
    long need = (work + work_items_per_block_iter - 1) / work_items_per_block_iter;
    long g = need < full ? need : full;
    return (int)(g < 1 ? 1 : g);
}

// grid of a memory-bound grid-stride kernel: enough blocks to fill the chip (`per_sm` resident blocks per SM) and no more --
// HBM likes a few hundred concurrent streams, not thousands (k_fft64<fast> at 5 blocks per SM: 5.7 TB/s, at 3: 6.5 TB/s)
int stream_grid(ofdm_ctx *ctx, long rows, int rows_per_block, int per_sm)
{
    const long need = (rows + rows_per_block - 1) / rows_per_block, full = (long)per_sm * ctx->sm_count;
    const long g = need < full ? need : full;
    return (int)(g < 1 ? 1 : g);
}

int ensure_scratch(ofdm_ctx *ctx, int slot, size_t bytes, void **out)
{
    if (ctx->scratch_bytes[slot] < bytes) {
        if (ctx->scratch[slot]) { cudaFree(ctx->scratch[slot]); ctx->scratch[slot] = nullptr; ctx->scratch_bytes[slot] = 0; }
        cudaError_t e = cudaMalloc(&ctx->scratch[slot], bytes);
        if (e != cudaSuccess) return fail(ctx, OFDM_ERR_NOMEM, "cudaMalloc(scratch)", e);
        ctx->scratch_bytes[slot] = bytes;
    }
    *out = ctx->scratch[slot];
    return OFDM_OK;
}

float snr_linear(float snr_db)
{
    // float snr_linear = pow(10, snr / 10);   OFDM.c:645  (float / int -> float, pow in double, rounded to float)
    return (float)pow(10.0, (double)(snr_db / 10));
}

// running float power sum of OFDM.c:637-641 over n samples, with the device's glibc-faithful hypot (one thread: the
// chain is sequential) -- the same arithmetic k_frame_power_exact continues from
__global__ void k_power_prefix(const float2 *__restrict__ x, int n, float *__restrict__ out)
{
    float p = 0.f;
    for (int i = 0; i < n; ++i) {
        const double h = hypot_glibc((double)x[i].x, (double)x[i].y);
        p = __double2float_rn(__dadd_rn((double)p, __dmul_rn(h, h)));
    }
    *out = p;
}

// __constant__ c_tab is per device, not per context: it is written once per device (first context), under this
// mutex, before any other context of that device can exist -- a later ofdm_ctx_create never touches it, so it cannot
// disturb kernels another context has in flight.  The host-side copies of the preambles are cached alongside.
struct DeviceTables {
    bool ready = false;
    float lts_freq[128], lts_time[320], sts_time[320], lts_power_prefix;
};
std::mutex g_tables_mutex;
DeviceTables g_tables[64];

int upload_tables(ofdm_ctx *ctx, const float *lts_time /* nullable */, float power_prefix)
{
    Tables t;
    memset(&t, 0, sizeof t);
    for (int k = 0; k < 32; ++k) t.tw64[k] = make_double2(kTw64[k][0], kTw64[k][1]);
    for (int k = 0; k < 64; ++k) {
        double a = 2.0 * 3.14159265358979323846 * k / 64.0;
        t.tw64f[k] = make_float2((float)cos(a), (float)(-sin(a)));
    }
    // centred index c -> data index (runs of OFDM.c:528-547): c = 6..10, 12..24, 26..31, 33..38, 40..52, 54..58
    signed char by_c[64];
    for (int c = 0; c < 64; ++c) by_c[c] = -1;
    const int lo[6] = {6, 12, 26, 33, 40, 54}, hi[6] = {10, 24, 31, 38, 52, 58};
    int d = 0;
    for (int r = 0; r < 6; ++r) for (int c = lo[r]; c <= hi[r]; ++c) by_c[c] = (signed char)d++;
    by_c[11] = -2; by_c[25] = -2; by_c[39] = -2; by_c[53] = -3;           // pilots {1,1,1,-1} OFDM.c:523
    for (int p = 0; p < 64; ++p) {
        int c = (p + 32) & 63;
        t.bin_data[p] = by_c[c];
        t.bin_lts[p] = (c >= 6 && c <= 58) ? kLk[c - 6] : 0;
        if (by_c[c] >= 0) t.data_bin[by_c[c]] = (int8_t)p;
    }
    if (lts_time) {
        memcpy(t.lts_time, lts_time, sizeof t.lts_time);
        double sum = 0.0;
        for (int i = 0; i < 160; ++i) sum += (double)lts_time[2 * i] * lts_time[2 * i] + (double)lts_time[2 * i + 1] * lts_time[2 * i + 1];
        t.lts_power_prefix = power_prefix;        // OFDM.c:637-641 over the LTS slot, computed on the device (k_power_prefix)
        t.lts_power_sum = (float)sum;
    }
    OFDM_CUDA(ctx, cudaMemcpyToSymbolAsync(c_tab, &t, sizeof t, 0, cudaMemcpyHostToDevice, ctx->stream));
    OFDM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return OFDM_OK;
}

template <bool EXACT, bool INV>
int launch_fft(ofdm_ctx *ctx, const float *in, float *out, long n)
{
    auto k = k_fft64<EXACT, INV>;
    int grid = grid_for(ctx, k, 0, kWarpsPerBlock * 4, n);
    const int cap = stream_grid(ctx, n, kWarpsPerBlock * 4, 3);       // the fp32 variants' registers would allow 5 blocks per SM
    if (grid > cap) grid = cap;
    k<<<grid, kThreads, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(in), reinterpret_cast<float2 *>(out), n);
    return check_launch(ctx, "k_fft64");
}

// persistent launch of a kernel that takes one params struct with n_frames: blocks of `warps` warps, a warp on `per_warp` frames
// at a time
template <typename K, typename P>
int launch_persistent(ofdm_ctx *ctx, K k, int warps, int per_warp, size_t smem, const P &p, const char *name)
{
    if (smem) OFDM_CUDA(ctx, allow_smem(ctx, k, smem));
    const int grid = grid_for(ctx, k, smem, (long)warps * per_warp, p.n_frames, warps * 32);
    k<<<grid, warps * 32, smem, ctx->stream>>>(p);
    return check_launch(ctx, name);
}

// runtime noise source / arithmetic -> template argument: f(std::integral_constant<int, value>)
template <typename F>
int with_noise(int noise, F f)
{
    if (noise == kNoiseNone) return f(std::integral_constant<int, kNoiseNone>());
    if (noise == kNoiseInject) return f(std::integral_constant<int, kNoiseInject>());
    return f(std::integral_constant<int, kNoisePhilox>());
}
template <typename F>
int with_arith(int arith, F f)
{
    if (arith == kArithFast) return f(std::integral_constant<int, kArithFast>());
    if (arith == kArithChecked) return f(std::integral_constant<int, kArithChecked>());
    return f(std::integral_constant<int, kArithExact>());
}

// EXACT speculates in fp32, verifies and replays exactly (kArithChecked) unless "exact_speculation" = 0
int arith_of(const ofdm_ctx *ctx, int mode) { return mode != OFDM_MODE_EXACT ? kArithFast : ctx->checked ? kArithChecked : kArithExact; }

enum { kRxQuad, kRxN, kRx2, kRxGeneric };

// receiver family: the streaming kernels need no per-bin outputs and 16-byte aligned buffers (bulk copies); one frame per lane
// group (k_stream_quad, ofdm_stream.cuh) for the speculating arithmetic, else one frame per warp -- the multi-pass kernel for
// other frame shapes (or "general_stream" = 1), k_stream_rx2 for the default one
int rx_family(const ofdm_ctx *ctx, int arith, int noise, const RxParams &p, bool dump)
{
    const bool aligned = ((uintptr_t)p.in % 16 == 0) && (noise != kNoiseInject || (uintptr_t)p.g % 16 == 0);
    if (dump || !aligned || ctx->force_generic) return kRxGeneric;
    if (ctx->stream_layout == 0 && arith != kArithExact) return kRxQuad;
    return p.n_sym != 2 || ctx->general_stream ? kRxN : kRx2;
}

// arithmetic policy of the streaming receivers: the all-exact kernels take the caller's params; the speculating ones get the
// error radii (ofdm_chain.cuh: kRadius, kChanRadius) and the EVM guard (fast mode: tiny |H| bins are replayed exactly), except
// fp32 with Philox noise, whose results are statistical: plain fp32 like the fused Monte-Carlo kernel
RxParams rx_policy(const ofdm_ctx *ctx, int arith, int noise, RxParams q)
{
    if (arith == kArithExact) return q;
    q.replayed = ctx->replayed_dev;
    q.evm_guard = arith == kArithFast && noise == kNoisePhilox ? 0.f : ctx->evm_guard;
    q.radius_scale = ctx->force_replay ? INFINITY : kRadius;
    q.radius_chan = ctx->force_replay ? INFINITY : kChanRadius * sqrtf((float)OFDM_FRAME_LEN(q.n_sym) * q.snr_lin) * 1.001f;
    return q;
}

int launch_rx_any(ofdm_ctx *ctx, int mode, int noise, const RxParams &p)
{
    const ofdm_rx_dump &d = p.dump;
    const bool dump = d.H || d.eq || d.sliced || d.bits || d.frame_bit_errors || d.frame_evm_lin;
    const int arith = arith_of(ctx, mode), family = rx_family(ctx, arith, noise, p, dump);
    if (family == kRxGeneric)           // the generic kernel takes the caller's params in both modes
        return with_noise(noise, [&](auto n) -> int {
            constexpr int N = decltype(n)::value;
            auto go = [&](auto k) { return launch_persistent(ctx, k, kWarpsPerBlock, 1, 0, p, "k_rx_frames"); };
            if (mode == OFDM_MODE_EXACT) return dump ? go(k_rx_frames<true, N, true>) : go(k_rx_frames<true, N, false>);
            return dump ? go(k_rx_frames<false, N, true>) : go(k_rx_frames<false, N, false>);
        });
    const RxParams q = rx_policy(ctx, arith, noise, p);
    return with_noise(noise, [&](auto n) -> int {
        return with_arith(arith, [&](auto a) -> int {
            constexpr int N = decltype(n)::value, A = decltype(a)::value;
            if constexpr (A != kArithExact) {
                if (family == kRxQuad) {
                    auto go = [&](auto k, int warps) { return launch_persistent(ctx, k, warps, 4, quad_smem_bytes<N>(warps), q, "k_stream_quad"); };
                    if (ctx->stream_warps == 8) return go(k_stream_quad<A, N, 8>, 8);
                    // the default frame shape has its own build: unit w of a quad always in ring slot w ("general_stream" = 1 keeps the general one)
                    if (p.n_sym == 2 && !ctx->general_stream) return go(k_stream_quad<A, N, 6, true>, 6);
                    return go(k_stream_quad<A, N, 6>, 6);
                }
            }
            if (family == kRxN) return launch_persistent(ctx, k_stream_rxn<A, N>, kWarpsPerBlock, 1, stream_smem_bytes<N>(), q, "k_stream_rxn");
            return launch_persistent(ctx, k_stream_rx2<A, N>, kWarpsPerBlock, 1, stream_smem_bytes<N>(), q, "k_stream_rx2");
        });
    });
}

int blocks_1d(long n) { return (int)((n + 255) / 256); }

int frame_power(ofdm_ctx *ctx, const float *frames, float *power, long n_frames, int len, int mode, bool lts_prefix = false)
{
    if (mode == OFDM_MODE_EXACT) {
        // frames straight from the transmitter start with the LTS slot, whose partial sum is a build constant
        const bool vec_ok = ((uintptr_t)frames % 16 == 0) && (len % 2 == 0);
        const bool skip = lts_prefix && vec_ok;
        const float2 *x = reinterpret_cast<const float2 *>(frames);
        const int first = skip ? 160 : 0;
        if (vec_ok && (len - first) % 16 == 0 && len > first)
            k_frame_power_tiled<<<(int)((n_frames + 255) / 256), kThreads, 0, ctx->stream>>>(x, power, n_frames, len, first,
                                                                                           skip ? ctx->lts_power_prefix : 0.0f, ctx->power_margin);
        else if (vec_ok)
            k_frame_power_exact<true><<<blocks_1d(n_frames), 256, 0, ctx->stream>>>(x, power, n_frames, len, skip ? 160 : 0,
                                                                                  skip ? ctx->lts_power_prefix : 0.0f);
        else
            k_frame_power_exact<false><<<blocks_1d(n_frames), 256, 0, ctx->stream>>>(x, power, n_frames, len, 0, 0.0f);
        return check_launch(ctx, "k_frame_power_exact");
    }
    int grid = grid_for(ctx, k_frame_power_fast, 0, kWarpsPerBlock, n_frames);
    k_frame_power_fast<<<grid, kThreads, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(frames), power, n_frames, len);
    return check_launch(ctx, "k_frame_power_fast");
}

// Channel + receiver of a whole SNR list on resident frames: the all-SNR kernel when it applies (two-symbol frames, 16-byte
// aligned buffers, speculation allowed), else one fused channel+receiver launch per SNR point.  counters [n_snr], accumulated into.
int sweep_points(ofdm_ctx *ctx, const float *frames, const float *g, const float *power, const uint32_t *bits, long n_frames, int n_sym,
                 const float *snr_db, int n_snr, int mode, ofdm_counters *counters);

bool mode_ok(int mode) { return mode == OFDM_MODE_EXACT || mode == OFDM_MODE_FAST; }
bool nsym_ok(int n_sym) { return n_sym >= 1 && n_sym <= OFDM_MAX_SYM; }
bool noise_ok(int noise) { return noise == OFDM_NOISE_REAL_RAIL || noise == OFDM_NOISE_COMPLEX; }
bool snr_def_ok(int snr_def) { return snr_def >= OFDM_SNR_FRAME_POWER && snr_def <= OFDM_SNR_EBN0; }
bool is_reference_channel(int noise, int snr_def) { return noise == OFDM_NOISE_REAL_RAIL && snr_def == OFDM_SNR_FRAME_POWER; }

// noise power of an Es/N0 or Eb/N0 point: a data bin carries X (|X| = 1) and, through the transmitter's 1/64 IFFT and the
// receiver's unscaled FFT, noise of variance 64 np, so Es/N0 = 1 / (64 np); Eb/N0 = Es/N0 / bits, bits = the information bits
// a QPSK point carries (2 uncoded, 2R behind a rate-R code; the 6 tail bits are not counted).  In double, rounded to float once.
float fixed_noise_power(int snr_def, float snr_db, double bits = 2.0)
{
    const double per_point = snr_def == OFDM_SNR_EBN0 ? 64.0 * bits : 64.0;
    return (float)(1.0 / (per_point * pow(10.0, (double)snr_db / 10.0)));
}

// k_awgn_channel over n_frames frames of len samples: power != NULL -> np = power[f] / snr_lin, else np = np_fixed
int launch_awgn_channel(ofdm_ctx *ctx, int noise, const float *tx, const float *power, float snr_lin, float np_fixed, uint32_t seed,
                        uint32_t stream, uint64_t frame0, float *ota, long n_frames, int len, int mode)
{
    const float2 *x = reinterpret_cast<const float2 *>(tx);
    float2 *y = reinterpret_cast<float2 *>(ota);
    auto launch = [&](auto k) -> int {
        int grid = grid_for(ctx, k, 0, kWarpsPerBlock, n_frames);
        k<<<grid, kThreads, 0, ctx->stream>>>(x, power, snr_lin, np_fixed, seed, stream, frame0, y, n_frames, len);
        return check_launch(ctx, "k_awgn_channel");
    };
    const bool cx = noise == OFDM_NOISE_COMPLEX;
    if (mode == OFDM_MODE_EXACT) return cx ? launch(k_awgn_channel<true, true>) : launch(k_awgn_channel<true, false>);
    return cx ? launch(k_awgn_channel<false, true>) : launch(k_awgn_channel<false, false>);
}

bool rate_ok(int rate) { return rate == OFDM_CODE_R12 || rate == OFDM_CODE_R34; }
bool code_ok(const ofdm_code *code)
{
    return code != nullptr && rate_ok(code->rate) && (code->decision == OFDM_DECISION_SOFT || code->decision == OFDM_DECISION_HARD);
}
// information bits per QPSK point: 2 uncoded, 2R behind the code
double info_bits_per_point(const ofdm_code *code) { return code == nullptr ? 2.0 : code->rate == OFDM_CODE_R12 ? 1.0 : 1.5; }

int launch_conv_encode(ofdm_ctx *ctx, int rate, const uint32_t *info, uint32_t *payload, long n_frames, int n_sym)
{
    auto k = rate == OFDM_CODE_R12 ? k_conv_encode<kCodeR12> : k_conv_encode<kCodeR34>;
    k<<<blocks_1d(n_frames * n_sym), 256, 0, ctx->stream>>>(info, payload, n_frames, n_sym);
    return check_launch(ctx, "k_conv_encode");
}

// k_viterbi over n_frames frames: a block's survivors stay in shared memory up to kVitSmemMax (two-symbol frames: 6 KB at rate
// 1/2, 9 KB at 3/4), longer frames keep them in a scratch buffer in HBM for a grid of at most two blocks per SM (the longest
// frames: 288 KiB per warp).  Same code either way, so the same bits.  One launch per 2^20 frames: the per-lane totals are 32-bit.
int launch_viterbi(ofdm_ctx *ctx, const ofdm_code &code, const float *H, const float *eq, const uint32_t *info, uint32_t *decoded,
                   long n_frames, int n_sym, ofdm_counters *counters)
{
    const size_t per_warp = vit_surv_bytes(code.rate, n_sym);
    const bool in_smem = per_warp * kVitWarps <= (size_t)kVitSmemMax;
    const size_t smem = in_smem ? per_warp * kVitWarps : 0;
    const long max_frames = 1L << 20;
    auto go = [&](auto k) -> int {
        if (in_smem) OFDM_CUDA(ctx, allow_smem(ctx, k, kVitSmemMax));
        for (long f0 = 0; f0 < n_frames; f0 += max_frames) {
            VitParams p;
            memset(&p, 0, sizeof p);
            p.n_frames = n_frames - f0 < max_frames ? n_frames - f0 : max_frames;
            p.n_sym = n_sym;
            p.H = reinterpret_cast<const float2 *>(H) + f0 * 64;
            p.eq = reinterpret_cast<const float2 *>(eq) + f0 * n_sym * 48;
            p.info = info ? info + f0 * n_sym * 3 : nullptr;
            p.decoded = decoded ? decoded + f0 * n_sym * 3 : nullptr;
            p.counters = counters;
            int grid = grid_for(ctx, k, smem, kVitWarps, p.n_frames, kVitWarps * 32);
            if (!in_smem) {
                if (grid > 2 * ctx->sm_count) grid = 2 * ctx->sm_count;
                void *buf = nullptr;
                if (int st = ensure_scratch(ctx, 10, (size_t)grid * kVitWarps * per_warp, &buf)) return st;
                p.surv_global = reinterpret_cast<uint2 *>(buf);
            }
            k<<<grid, kVitWarps * 32, smem, ctx->stream>>>(p);
            if (int st = check_launch(ctx, "k_viterbi")) return st;
        }
        return OFDM_OK;
    };
    const bool hard = code.decision == OFDM_DECISION_HARD;
    if (code.rate == OFDM_CODE_R12) return hard ? go(k_viterbi<kCodeR12, kDecisionHard>) : go(k_viterbi<kCodeR12, kDecisionSoft>);
    return hard ? go(k_viterbi<kCodeR34, kDecisionHard>) : go(k_viterbi<kCodeR34, kDecisionSoft>);
}


}  // namespace

extern "C" {

int ofdm_version(void) { return OFDM_B200_VERSION; }

const char *ofdm_strerror(int status)
{
    switch (status) {
    case OFDM_OK: return "ok";
    case OFDM_ERR_INVALID: return "invalid argument";
    case OFDM_ERR_CUDA: return "CUDA runtime error";
    case OFDM_ERR_NOMEM: return "out of memory";
    case OFDM_ERR_IO: return "file I/O error";
    case OFDM_ERR_NODEVICE: return "no CUDA device (this library has no CPU fallback)";
    default: return "unknown status";
    }
}

int ofdm_ctx_create(ofdm_ctx **out, int device)
{
    if (!out) return OFDM_ERR_INVALID;
    *out = nullptr;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev < 1) { cudaGetLastError(); return OFDM_ERR_NODEVICE; }
    if (device < 0 || device >= n_dev) return OFDM_ERR_INVALID;
    ofdm_ctx *ctx = new (std::nothrow) ofdm_ctx();
    if (!ctx) return OFDM_ERR_NOMEM;
    ctx->device = device;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete ctx; return OFDM_ERR_CUDA; }
    ctx->owns_stream = true;

    std::lock_guard<std::mutex> lock(g_tables_mutex);
    DeviceTables &dt = g_tables[device & 63];
    int st = OFDM_OK;
    float *d_buf = nullptr;
    if (dt.ready) {                 // the device's tables are in place: nothing is uploaded, nothing running is disturbed
        memcpy(ctx->lts_freq, dt.lts_freq, sizeof dt.lts_freq);
        memcpy(ctx->lts_time, dt.lts_time, sizeof dt.lts_time);
        memcpy(ctx->sts_time, dt.sts_time, sizeof dt.sts_time);
        ctx->lts_power_prefix = dt.lts_power_prefix;
    } else {
    // LTS: Preamble_Generator(type 1) OFDM.c:368-399 -- frequency grid from L_k at c = 6..58, time slot through
    // this library's own exact ifft kernel (it reads only the twiddles of c_tab), then [samples 32..63][0..63][0..63]
    st = upload_tables(ctx, nullptr, 0.f);
    if (st == OFDM_OK && cudaMalloc(&d_buf, (2 * 128 + 320 + 4) * sizeof(float)) != cudaSuccess) st = OFDM_ERR_NOMEM;
    if (st == OFDM_OK) {
        memset(ctx->lts_freq, 0, sizeof ctx->lts_freq);
        for (int i = 0; i < 53; ++i) ctx->lts_freq[2 * (6 + i)] = (float)kLk[i];
        float t64[128];
        if (cudaMemcpyAsync(d_buf, ctx->lts_freq, sizeof ctx->lts_freq, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) st = OFDM_ERR_CUDA;
        if (st == OFDM_OK) st = launch_fft<true, true>(ctx, d_buf, d_buf + 128, 1);
        if (st == OFDM_OK && cudaMemcpyAsync(t64, d_buf + 128, sizeof t64, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) st = OFDM_ERR_CUDA;
        if (st == OFDM_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) st = OFDM_ERR_CUDA;
        if (st == OFDM_OK) {
            memcpy(ctx->lts_time, t64 + 64, 32 * 2 * sizeof(float));                 // :396
            memcpy(ctx->lts_time + 64, t64, 64 * 2 * sizeof(float));                 // :397 (first copy)
            memcpy(ctx->lts_time + 64 + 128, t64, 64 * 2 * sizeof(float));           // :397 (second copy)
            // the exact-mode power prefix of the LTS slot, in the device's own arithmetic (the kernels continue this chain)
            float *d_lts = d_buf + 256, *d_pref = d_buf + 256 + 320;
            if (cudaMemcpyAsync(d_lts, ctx->lts_time, sizeof ctx->lts_time, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) st = OFDM_ERR_CUDA;
            if (st == OFDM_OK) {
                k_power_prefix<<<1, 1, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(d_lts), 160, d_pref);
                st = check_launch(ctx, "k_power_prefix");
            }
            if (st == OFDM_OK && cudaMemcpyAsync(&ctx->lts_power_prefix, d_pref, sizeof(float), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) st = OFDM_ERR_CUDA;
            if (st == OFDM_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) st = OFDM_ERR_CUDA;
            if (st == OFDM_OK) st = upload_tables(ctx, ctx->lts_time, ctx->lts_power_prefix);
        }
    }
    // STS: Preamble_Generator(type 0) OFDM.c:479-492: S_k * (float)sqrt(13/6) at c = 6..58, exact ifft, first 16 samples x 10 (:393)
    if (st == OFDM_OK) {
        static const signed char Sk[53] = {0,0,1,0,0,0,-1,0,0,0, 1,0,0,0,-1,0,0,0,-1,0,0,0, 1,0,0,0,0,0,0,0,-1,0,0,0, -1,0,0,0,1,0,0,0,1,0,0,0, 1,0,0,0,1,0,0};
        const float scale = (float)sqrt(13.0 / 6.0);
        float grid[128], t64[128];
        memset(grid, 0, sizeof grid);
        for (int i = 0; i < 53; ++i) { grid[2 * (6 + i)] = (float)Sk[i] * scale; grid[2 * (6 + i) + 1] = (float)Sk[i] * scale; }
        if (cudaMemcpyAsync(d_buf, grid, sizeof grid, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) st = OFDM_ERR_CUDA;
        if (st == OFDM_OK) st = launch_fft<true, true>(ctx, d_buf, d_buf + 128, 1);
        if (st == OFDM_OK && cudaMemcpyAsync(t64, d_buf + 128, sizeof t64, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) st = OFDM_ERR_CUDA;
        if (st == OFDM_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) st = OFDM_ERR_CUDA;
        if (st == OFDM_OK) for (int r = 0; r < 10; ++r) memcpy(ctx->sts_time + 32 * r, t64, 16 * 2 * sizeof(float));
    }
    if (st == OFDM_OK) {
        memcpy(dt.lts_freq, ctx->lts_freq, sizeof dt.lts_freq);
        memcpy(dt.lts_time, ctx->lts_time, sizeof dt.lts_time);
        memcpy(dt.sts_time, ctx->sts_time, sizeof dt.sts_time);
        dt.lts_power_prefix = ctx->lts_power_prefix;
        dt.ready = true;
    }
    }
    if (st == OFDM_OK) {
        if (cudaMalloc(&ctx->replayed_dev, sizeof(unsigned long long)) != cudaSuccess) st = OFDM_ERR_NOMEM;
        else if (cudaMemset(ctx->replayed_dev, 0, sizeof(unsigned long long)) != cudaSuccess) st = OFDM_ERR_CUDA;
    }
    if (st == OFDM_OK) {            // per-context device copy of the STS slot (ofdm_prepend_sts)
        if (cudaMalloc(&ctx->sts_dev, sizeof ctx->sts_time) != cudaSuccess) st = OFDM_ERR_NOMEM;
        else if (cudaMemcpy(ctx->sts_dev, ctx->sts_time, sizeof ctx->sts_time, cudaMemcpyHostToDevice) != cudaSuccess) st = OFDM_ERR_CUDA;
    }
    if (d_buf) cudaFree(d_buf);
    if (st != OFDM_OK) { ofdm_ctx_destroy(ctx); return st; }
    *out = ctx;
    return OFDM_OK;
}

int ofdm_ctx_destroy(ofdm_ctx *ctx)
{
    if (!ctx) return OFDM_ERR_INVALID;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < 11; ++i) if (ctx->scratch[i]) cudaFree(ctx->scratch[i]);
    if (ctx->sts_dev) cudaFree(ctx->sts_dev);
    if (ctx->replayed_dev) cudaFree(ctx->replayed_dev);
    if (ctx->copy_stream) {
        cudaStreamSynchronize(ctx->copy_stream);
        cudaStreamDestroy(ctx->copy_stream);
        for (int i = 0; i < 2; ++i) cudaEventDestroy(ctx->copy_done[i]);
        cudaEventDestroy(ctx->call_start);
    }
    if (ctx->owns_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return OFDM_OK;
}

const char *ofdm_last_error(const ofdm_ctx *ctx) { return ctx ? ctx->err : "null context"; }

int ofdm_ctx_set_stream(ofdm_ctx *ctx, void *cuda_stream)
{
    if (!ctx) return OFDM_ERR_INVALID;
    if (ctx->owns_stream && ctx->stream) { cudaStreamSynchronize(ctx->stream); cudaStreamDestroy(ctx->stream); }
    ctx->stream = (cudaStream_t)cuda_stream;
    ctx->owns_stream = false;
    return OFDM_OK;
}
void *ofdm_ctx_stream(const ofdm_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
int ofdm_ctx_sync(ofdm_ctx *ctx)
{
    if (int st = bind(ctx)) return st;
    OFDM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return OFDM_OK;
}
int ofdm_ctx_set_option(ofdm_ctx *ctx, const char *name, int value)
{
    if (!ctx || !name) return OFDM_ERR_INVALID;
    if (!strcmp(name, "force_generic_rx")) { ctx->force_generic = value != 0; return OFDM_OK; }
    if (!strcmp(name, "exact_speculation")) { ctx->checked = value != 0; return OFDM_OK; }
    if (!strcmp(name, "force_replay")) { ctx->force_replay = value != 0; return OFDM_OK; }
    if (!strcmp(name, "evm_guard")) { if (value < 1 || value > 65536) return fail(ctx, OFDM_ERR_INVALID, "evm_guard: 1..65536 radii"); ctx->evm_guard = (float)value; return OFDM_OK; }
    if (!strcmp(name, "power_margin")) { if (value < 16 || value > (1 << 28)) return fail(ctx, OFDM_ERR_INVALID, "power_margin: 16..2^28 ulps"); ctx->power_margin = (uint32_t)value; return OFDM_OK; }
    if (!strcmp(name, "fused_sweep")) { ctx->fused_sweep = value != 0; return OFDM_OK; }
    if (!strcmp(name, "general_stream")) { ctx->general_stream = value != 0; return OFDM_OK; }
    if (!strcmp(name, "stream_warps")) { if (value != 6 && value != 8) return fail(ctx, OFDM_ERR_INVALID, "stream_warps: 6 or 8"); ctx->stream_warps = value; return OFDM_OK; }
    if (!strcmp(name, "stream_layout")) { if (value < 0 || value > 1) return fail(ctx, OFDM_ERR_INVALID, "stream_layout: 0..1"); ctx->stream_layout = value; return OFDM_OK; }
    if (!strcmp(name, "multipath_path")) { if (value < 0 || value > 2) return fail(ctx, OFDM_ERR_INVALID, "multipath_path: 0..2"); ctx->multipath_path = value; return OFDM_OK; }
    return fail(ctx, OFDM_ERR_INVALID, "unknown option");
}
int ofdm_ctx_replayed_frames(ofdm_ctx *ctx, uint64_t *count, int reset)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, count != nullptr);
    unsigned long long v = 0;
    OFDM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    OFDM_CUDA(ctx, cudaMemcpy(&v, ctx->replayed_dev, sizeof v, cudaMemcpyDeviceToHost));
    *count = v;
    if (reset) OFDM_CUDA(ctx, cudaMemset(ctx->replayed_dev, 0, sizeof v));
    return OFDM_OK;
}
int ofdm_ctx_sm_count(const ofdm_ctx *ctx) { return ctx ? ctx->sm_count : 0; }
uint64_t ofdm_ctx_launch_count(const ofdm_ctx *ctx) { return ctx ? ctx->launches : 0; }

int ofdm_dev_alloc(ofdm_ctx *ctx, void **ptr, size_t bytes)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, ptr != nullptr);
    cudaError_t e = cudaMalloc(ptr, bytes ? bytes : 1);
    if (e != cudaSuccess) { *ptr = nullptr; return fail(ctx, OFDM_ERR_NOMEM, "cudaMalloc", e); }
    return OFDM_OK;
}
int ofdm_dev_free(ofdm_ctx *ctx, void *ptr)
{
    if (int st = bind(ctx)) return st;
    OFDM_CUDA(ctx, cudaFree(ptr));
    return OFDM_OK;
}
int ofdm_host_alloc(ofdm_ctx *ctx, void **ptr, size_t bytes)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, ptr != nullptr);
    cudaError_t e = cudaMallocHost(ptr, bytes ? bytes : 1);
    if (e != cudaSuccess) { *ptr = nullptr; return fail(ctx, OFDM_ERR_NOMEM, "cudaMallocHost", e); }
    return OFDM_OK;
}
int ofdm_host_free(ofdm_ctx *ctx, void *ptr)
{
    if (int st = bind(ctx)) return st;
    OFDM_CUDA(ctx, cudaFreeHost(ptr));
    return OFDM_OK;
}
int ofdm_memcpy_h2d(ofdm_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    if (int st = bind(ctx)) return st;
    if (bytes == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, dst != nullptr && src != nullptr);
    OFDM_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return OFDM_OK;
}
int ofdm_memcpy_d2h(ofdm_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    if (int st = bind(ctx)) return st;
    if (bytes == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, dst != nullptr && src != nullptr);
    OFDM_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return OFDM_OK;
}
int ofdm_memset_dev(ofdm_ctx *ctx, void *dst, int value, size_t bytes)
{
    if (int st = bind(ctx)) return st;
    if (bytes == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, dst != nullptr);
    OFDM_CUDA(ctx, cudaMemsetAsync(dst, value, bytes, ctx->stream));
    return OFDM_OK;
}

// ------------------------------------------------------------------ stage-level
int ofdm_pack_bits(ofdm_ctx *ctx, const uint8_t *bits, uint32_t *packed, long n_symbols)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_symbols >= 0);
    if (n_symbols == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, bits != nullptr && packed != nullptr);
    long n_words = n_symbols * 3;
    k_pack_bits<<<blocks_1d(n_words), 256, 0, ctx->stream>>>(bits, packed, n_words);
    return check_launch(ctx, "k_pack_bits");
}
int ofdm_unpack_bits(ofdm_ctx *ctx, const uint32_t *packed, uint8_t *bits, long n_symbols)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_symbols >= 0);
    if (n_symbols == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, bits != nullptr && packed != nullptr);
    long n_bits = n_symbols * 96;
    k_unpack_bits<<<blocks_1d(n_bits), 256, 0, ctx->stream>>>(packed, bits, n_bits);
    return check_launch(ctx, "k_unpack_bits");
}
int ofdm_qpsk_modulate(ofdm_ctx *ctx, const uint32_t *bits, float *mod, long n_symbols)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_symbols >= 0);
    if (n_symbols == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, bits != nullptr && mod != nullptr);
    if ((uintptr_t)mod % 16 == 0)
        k_qpsk_mod2<<<stream_grid(ctx, n_symbols, 2 * kRows4, 6), 2 * kRows4 * 24, 0, ctx->stream>>>(bits, reinterpret_cast<float4 *>(mod), n_symbols);
    else
        k_qpsk_mod<<<stream_grid(ctx, n_symbols, kRows4, 6), kRows4 * 48, 0, ctx->stream>>>(bits, reinterpret_cast<float2 *>(mod), n_symbols);
    return check_launch(ctx, "k_qpsk_mod");
}
int ofdm_map_subcarriers(ofdm_ctx *ctx, const float *mod, float *grid, long n_symbols)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_symbols >= 0);
    if (n_symbols == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, mod != nullptr && grid != nullptr);
    k_map_subcarriers<<<stream_grid(ctx, n_symbols, kRows4, 4), kRows4 * 64, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(mod), reinterpret_cast<float2 *>(grid), n_symbols);
    return check_launch(ctx, "k_map_subcarriers");
}
int ofdm_ifft64(ofdm_ctx *ctx, const float *in, float *out, long n, int mode)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n >= 0 && mode_ok(mode));
    if (n == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, in != nullptr && out != nullptr && in != out);
    return mode == OFDM_MODE_EXACT ? launch_fft<true, true>(ctx, in, out, n) : launch_fft<false, true>(ctx, in, out, n);
}
int ofdm_fft64(ofdm_ctx *ctx, const float *in, float *out, long n, int mode)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n >= 0 && mode_ok(mode));
    if (n == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, in != nullptr && out != nullptr && in != out);
    return mode == OFDM_MODE_EXACT ? launch_fft<true, false>(ctx, in, out, n) : launch_fft<false, false>(ctx, in, out, n);
}
int ofdm_add_cp(ofdm_ctx *ctx, const float *sym, float *out, long n)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n >= 0);
    if (n == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, sym != nullptr && out != nullptr);
    k_add_cp<<<stream_grid(ctx, n, kRows4, 4), kRows4 * 80, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(sym), reinterpret_cast<float2 *>(out), n);
    return check_launch(ctx, "k_add_cp");
}
int ofdm_lts(ofdm_ctx *ctx, float *lts_freq_host, float *lts_time_host)
{
    if (!ctx) return OFDM_ERR_INVALID;
    if (lts_freq_host) memcpy(lts_freq_host, ctx->lts_freq, sizeof ctx->lts_freq);
    if (lts_time_host) memcpy(lts_time_host, ctx->lts_time, sizeof ctx->lts_time);
    return OFDM_OK;
}

int ofdm_frame_power(ofdm_ctx *ctx, const float *frames, float *power, long n_frames, int frame_len, int mode)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && frame_len >= 1 && frame_len <= OFDM_FRAME_LEN(OFDM_MAX_SYM) && mode_ok(mode));
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, frames != nullptr && power != nullptr);
    return frame_power(ctx, frames, power, n_frames, frame_len, mode);
}

int ofdm_tx_frames(ofdm_ctx *ctx, const uint32_t *bits, float *frames, float *power, long n_frames, int n_sym, int mode)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && mode_ok(mode));
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, bits != nullptr && frames != nullptr);
    int st;
    if (n_sym == 2 && (uintptr_t)frames % 16 == 0 && !ctx->force_generic) {
        // default frame shape: frames leave shared memory through the TMA engine (k_tx_frames2)
        const size_t smem = tx2_smem_bytes();
        auto launch = [&](auto k) -> int {
            OFDM_CUDA(ctx, allow_smem(ctx, k, smem));
            int grid = grid_for(ctx, k, smem, kWarpsPerBlock * 2, n_frames);
            k<<<grid, kThreads, smem, ctx->stream>>>(bits, reinterpret_cast<float2 *>(frames), n_frames);
            return check_launch(ctx, "k_tx_frames2");
        };
        st = mode == OFDM_MODE_EXACT ? launch(k_tx_frames2<true>) : launch(k_tx_frames2<false>);
    } else if (mode == OFDM_MODE_EXACT) {
        int grid = grid_for(ctx, k_tx_frames<true>, 0, kWarpsPerBlock * 4, n_frames * n_sym);
        k_tx_frames<true><<<grid, kThreads, 0, ctx->stream>>>(bits, reinterpret_cast<float2 *>(frames), n_frames, n_sym);
        st = check_launch(ctx, "k_tx_frames<exact>");
    } else {
        int grid = grid_for(ctx, k_tx_frames<false>, 0, kWarpsPerBlock * 4, n_frames * n_sym);
        k_tx_frames<false><<<grid, kThreads, 0, ctx->stream>>>(bits, reinterpret_cast<float2 *>(frames), n_frames, n_sym);
        st = check_launch(ctx, "k_tx_frames<fast>");
    }
    if (st != OFDM_OK || power == nullptr) return st;
    return frame_power(ctx, frames, power, n_frames, OFDM_FRAME_LEN(n_sym), mode, true);
}

static int resolve_power(ofdm_ctx *ctx, const float *tx, const float *power, long n_frames, int len, int mode, const float **out)
{
    if (power) { *out = power; return OFDM_OK; }
    void *buf = nullptr;
    if (int st = ensure_scratch(ctx, 0, (size_t)n_frames * sizeof(float), &buf)) return st;
    if (int st = frame_power(ctx, tx, (float *)buf, n_frames, len, mode)) return st;
    *out = (const float *)buf;
    return OFDM_OK;
}

static int awgn_common(ofdm_ctx *ctx, int noise, const float *tx, const float *g, const float *power, float snr_db,
                       uint32_t seed, uint32_t stream, uint64_t frame0, float *ota, long n_frames, int n_sym, int mode)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && mode_ok(mode));
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, tx != nullptr && ota != nullptr && (noise != kNoiseInject || g != nullptr));
    const int len = OFDM_FRAME_LEN(n_sym);
    const float *pw = nullptr;
    if (int st = resolve_power(ctx, tx, power, n_frames, len, mode, &pw)) return st;
    const float2 *x = reinterpret_cast<const float2 *>(tx);
    float2 *y = reinterpret_cast<float2 *>(ota);
    const float sl = snr_linear(snr_db);
#define LAUNCH_AWGN(E, N)                                                                                         \
    do {                                                                                                          \
        int grid = grid_for(ctx, k_awgn<E, N>, 0, kWarpsPerBlock, n_frames);                                      \
        k_awgn<E, N><<<grid, kThreads, 0, ctx->stream>>>(x, g, pw, sl, seed, stream, frame0, y, n_frames, len);   \
    } while (0)
    if (mode == OFDM_MODE_EXACT) { if (noise == kNoiseInject) LAUNCH_AWGN(true, kNoiseInject); else LAUNCH_AWGN(true, kNoisePhilox); }
    else { if (noise == kNoiseInject) LAUNCH_AWGN(false, kNoiseInject); else LAUNCH_AWGN(false, kNoisePhilox); }
#undef LAUNCH_AWGN
    return check_launch(ctx, "k_awgn");
}

int ofdm_awgn_inject(ofdm_ctx *ctx, const float *tx, const float *g, const float *power, float snr_db, float *ota,
                     long n_frames, int n_sym, int mode)
{
    return awgn_common(ctx, kNoiseInject, tx, g, power, snr_db, 0, 0, 0, ota, n_frames, n_sym, mode);
}
int ofdm_awgn_philox(ofdm_ctx *ctx, const float *tx, const float *power, float snr_db, uint32_t seed, uint32_t stream,
                     uint64_t frame0, float *ota, long n_frames, int n_sym, int mode)
{
    return awgn_common(ctx, kNoisePhilox, tx, nullptr, power, snr_db, seed, stream, frame0, ota, n_frames, n_sym, mode);
}
int ofdm_awgn_philox_ex(ofdm_ctx *ctx, int noise, int snr_def, const float *tx, const float *power, float snr_db, uint32_t seed,
                        uint32_t stream, uint64_t frame0, float *ota, long n_frames, int n_sym, int mode)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, noise_ok(noise) && snr_def_ok(snr_def));
    if (is_reference_channel(noise, snr_def))
        return awgn_common(ctx, kNoisePhilox, tx, nullptr, power, snr_db, seed, stream, frame0, ota, n_frames, n_sym, mode);
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && mode_ok(mode));
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, tx != nullptr && ota != nullptr);
    const int len = OFDM_FRAME_LEN(n_sym);
    if (snr_def != OFDM_SNR_FRAME_POWER)
        return launch_awgn_channel(ctx, noise, tx, nullptr, 1.f, fixed_noise_power(snr_def, snr_db), seed, stream, frame0, ota, n_frames, len, mode);
    const float *pw = nullptr;
    if (int st = resolve_power(ctx, tx, power, n_frames, len, mode, &pw)) return st;
    return launch_awgn_channel(ctx, noise, tx, pw, snr_linear(snr_db), 0.f, seed, stream, frame0, ota, n_frames, len, mode);
}

static int rx_common(ofdm_ctx *ctx, int noise, const float *in, const float *g, const float *power, const uint32_t *tx_bits,
                     float snr_db, uint32_t seed, uint32_t stream, uint64_t frame0, long n_frames, int n_sym, int mode,
                     ofdm_counters *counters, const ofdm_rx_dump *dump)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && mode_ok(mode));
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, in != nullptr && tx_bits != nullptr && (noise != kNoiseInject || g != nullptr));
    RxParams p;
    memset(&p, 0, sizeof p);
    p.in = reinterpret_cast<const float2 *>(in);
    p.g = g;
    p.tx_bits = tx_bits;
    p.n_frames = n_frames;
    p.n_sym = n_sym;
    p.snr_lin = snr_linear(snr_db);
    p.seed = seed; p.stream = stream; p.frame0 = frame0;
    p.counters = counters;
    if (dump) p.dump = *dump;
    if (noise != kNoiseNone) {
        if (int st = resolve_power(ctx, in, power, n_frames, OFDM_FRAME_LEN(n_sym), mode, &p.power)) return st;
    }
    return launch_rx_any(ctx, mode, noise, p);
}

int ofdm_rx_frames(ofdm_ctx *ctx, const float *ota, const uint32_t *tx_bits, long n_frames, int n_sym, int mode,
                   ofdm_counters *counters, const ofdm_rx_dump *dump)
{
    return rx_common(ctx, kNoiseNone, ota, nullptr, nullptr, tx_bits, 0.f, 0, 0, 0, n_frames, n_sym, mode, counters, dump);
}
int ofdm_awgn_rx_inject(ofdm_ctx *ctx, const float *tx, const float *g, const float *power, const uint32_t *tx_bits,
                        float snr_db, long n_frames, int n_sym, int mode, ofdm_counters *counters, const ofdm_rx_dump *dump)
{
    return rx_common(ctx, kNoiseInject, tx, g, power, tx_bits, snr_db, 0, 0, 0, n_frames, n_sym, mode, counters, dump);
}
int ofdm_awgn_rx_philox(ofdm_ctx *ctx, const float *tx, const float *power, const uint32_t *tx_bits, float snr_db,
                        uint32_t seed, uint32_t stream, uint64_t frame0, long n_frames, int n_sym, int mode,
                        ofdm_counters *counters, const ofdm_rx_dump *dump)
{
    return rx_common(ctx, kNoisePhilox, tx, nullptr, power, tx_bits, snr_db, seed, stream, frame0, n_frames, n_sym, mode,
                     counters, dump);
}

int ofdm_awgn_rx_inject_sweep(ofdm_ctx *ctx, const float *tx, const float *g, const float *power, const uint32_t *tx_bits, const float *snr_db,
                              int n_snr, long n_frames, int n_sym, int mode, ofdm_counters *counters)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && mode_ok(mode) && n_snr >= 0);
    if (n_frames == 0 || n_snr == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, tx != nullptr && g != nullptr && tx_bits != nullptr && snr_db != nullptr && counters != nullptr);
    const float *pw = nullptr;
    if (int st = resolve_power(ctx, tx, power, n_frames, OFDM_FRAME_LEN(n_sym), mode, &pw)) return st;
    return sweep_points(ctx, tx, g, pw, tx_bits, n_frames, n_sym, snr_db, n_snr, mode, counters);
}

// ------------------------------------------------------------------ the receiver's stages one by one
int ofdm_strip_cp(ofdm_ctx *ctx, const float *frames, float *bodies, long n_frames, int n_sym, int frame_len, int data_off)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && data_off >= 0 && frame_len >= data_off + 80 * n_sym);
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, frames != nullptr && bodies != nullptr && frames != bodies);
    k_strip_cp<<<stream_grid(ctx, n_frames, kWarpsPerBlock, 4), kThreads, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(frames), reinterpret_cast<float2 *>(bodies), n_frames, n_sym, frame_len, data_off);
    return check_launch(ctx, "k_strip_cp");
}
int ofdm_channel_estimate(ofdm_ctx *ctx, const float *frames, float *H, long n_frames, int frame_len, int lts_off, int mode)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && mode_ok(mode) && lts_off >= 0 && frame_len >= lts_off + 160);
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, frames != nullptr && H != nullptr && frames != H);
    const float2 *x = reinterpret_cast<const float2 *>(frames);
    float2 *h = reinterpret_cast<float2 *>(H);
    if (mode == OFDM_MODE_EXACT) {
        int grid = grid_for(ctx, k_channel_estimate<true>, 0, kWarpsPerBlock * 2, n_frames);
        k_channel_estimate<true><<<grid, kThreads, 0, ctx->stream>>>(x, h, n_frames, frame_len, lts_off);
    } else {
        int grid = grid_for(ctx, k_channel_estimate<false>, 0, kWarpsPerBlock * 2, n_frames);
        k_channel_estimate<false><<<grid, kThreads, 0, ctx->stream>>>(x, h, n_frames, frame_len, lts_off);
    }
    return check_launch(ctx, "k_channel_estimate");
}
int ofdm_equalize(ofdm_ctx *ctx, const float *F, const float *H, float *E, long n_frames, int n_sym, int mode)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && mode_ok(mode));
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, F != nullptr && H != nullptr && E != nullptr);
    const int grid = stream_grid(ctx, n_frames, kWarpsPerBlock, 4);
    if (mode == OFDM_MODE_EXACT)
        k_equalize<true><<<grid, kThreads, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(F), reinterpret_cast<const float2 *>(H), reinterpret_cast<float2 *>(E), n_frames, n_sym);
    else
        k_equalize<false><<<grid, kThreads, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(F), reinterpret_cast<const float2 *>(H), reinterpret_cast<float2 *>(E), n_frames, n_sym);
    return check_launch(ctx, "k_equalize");
}
int ofdm_demap(ofdm_ctx *ctx, const float *grid, float *points, long n_symbols)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_symbols >= 0);
    if (n_symbols == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, grid != nullptr && points != nullptr && grid != points);
    k_demap<<<stream_grid(ctx, n_symbols, kRows4, 6), kRows4 * 48, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(grid), reinterpret_cast<float2 *>(points), n_symbols);
    return check_launch(ctx, "k_demap");
}
int ofdm_agc_slicer(ofdm_ctx *ctx, const float *points, float *sliced, long n_symbols)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_symbols >= 0);
    if (n_symbols == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, points != nullptr && sliced != nullptr);
    const long n = n_symbols * 48;
    if (((uintptr_t)points | (uintptr_t)sliced) % 16 == 0)            // n is even: 48 points per symbol
        k_agc_slicer2<<<stream_grid(ctx, n / 2, kThreads, 4), kThreads, 0, ctx->stream>>>(reinterpret_cast<const float4 *>(points), reinterpret_cast<float4 *>(sliced), n / 2);
    else
        k_agc_slicer<<<blocks_1d(n), 256, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(points), reinterpret_cast<float2 *>(sliced), n);
    return check_launch(ctx, "k_agc_slicer");
}
int ofdm_qpsk_demodulate(ofdm_ctx *ctx, const float *points, uint32_t *bits, long n_symbols)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_symbols >= 0);
    if (n_symbols == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, points != nullptr && bits != nullptr);
    const long n = n_symbols * 3;
    if ((uintptr_t)points % 16 == 0)
        k_qpsk_demod_warp<<<stream_grid(ctx, (n + 31) / 32, kWarpsPerBlock, 4), kThreads, 0, ctx->stream>>>(reinterpret_cast<const float4 *>(points), bits, n);
    else
        k_qpsk_demod<<<blocks_1d(n), 256, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(points), bits, n);
    return check_launch(ctx, "k_qpsk_demod");
}

// ------------------------------------------------------------------ sweep drivers
int ofdm_sweep_inject_dev(ofdm_ctx *ctx, const uint32_t *bits, const float *g, long n_frames, int n_sym,
                          const float *snr_db, int n_snr, int mode, ofdm_counters *out_host)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && mode_ok(mode) && n_snr >= 0);
    OFDM_REQUIRE(ctx, n_snr == 0 || (snr_db != nullptr && out_host != nullptr));
    if (n_snr > 0) memset(out_host, 0, sizeof(ofdm_counters) * (size_t)n_snr);
    if (n_frames == 0 || n_snr == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, bits != nullptr && g != nullptr);
    const int len = OFDM_FRAME_LEN(n_sym);
    void *frames = nullptr, *power = nullptr, *cnt = nullptr;
    if (int st = ensure_scratch(ctx, 1, (size_t)n_frames * len * 2 * sizeof(float), &frames)) return st;
    if (int st = ensure_scratch(ctx, 2, (size_t)n_frames * sizeof(float), &power)) return st;
    if (int st = ensure_scratch(ctx, 3, sizeof(ofdm_counters) * (size_t)n_snr, &cnt)) return st;
    OFDM_CUDA(ctx, cudaMemsetAsync(cnt, 0, sizeof(ofdm_counters) * (size_t)n_snr, ctx->stream));
    // Transmitter() runs once (OFDM.c:1191); the SNR loop (OFDM.c:1202-1222) reruns channel + receiver
    if (int st = ofdm_tx_frames(ctx, bits, (float *)frames, (float *)power, n_frames, n_sym, mode)) return st;
    if (int st = sweep_points(ctx, (const float *)frames, g, (const float *)power, bits, n_frames, n_sym, snr_db, n_snr, mode, (ofdm_counters *)cnt))
        return st;
    OFDM_CUDA(ctx, cudaMemcpyAsync(out_host, cnt, sizeof(ofdm_counters) * (size_t)n_snr, cudaMemcpyDeviceToHost, ctx->stream));
    OFDM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return OFDM_OK;
}

int ofdm_sweep_inject_host(ofdm_ctx *ctx, const uint32_t *bits_host, const float *g_host, long n_frames, int n_sym,
                           const float *snr_db, int n_snr, int mode, ofdm_counters *out_host)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && mode_ok(mode) && n_snr >= 0);
    if (n_frames == 0 || n_snr == 0) return ofdm_sweep_inject_dev(ctx, nullptr, nullptr, n_frames, n_sym, snr_db, n_snr, mode, out_host);
    OFDM_REQUIRE(ctx, bits_host != nullptr && g_host != nullptr && snr_db != nullptr && out_host != nullptr);
    const int len = OFDM_FRAME_LEN(n_sym);
    void *bits = nullptr, *g = nullptr, *frames = nullptr, *power = nullptr, *cnt = nullptr;
    const size_t bits_per_frame = (size_t)n_sym * 3 * sizeof(uint32_t), g_per_frame = (size_t)len * sizeof(float);
    if (int st = ensure_scratch(ctx, 4, (size_t)n_frames * bits_per_frame, &bits)) return st;
    if (int st = ensure_scratch(ctx, 5, (size_t)n_frames * g_per_frame, &g)) return st;
    if (int st = ensure_scratch(ctx, 1, (size_t)n_frames * len * 2 * sizeof(float), &frames)) return st;
    if (int st = ensure_scratch(ctx, 2, (size_t)n_frames * sizeof(float), &power)) return st;
    if (int st = ensure_scratch(ctx, 3, sizeof(ofdm_counters) * (size_t)n_snr, &cnt)) return st;
    if (!ctx->copy_stream) {
        OFDM_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) OFDM_CUDA(ctx, cudaEventCreateWithFlags(&ctx->copy_done[i], cudaEventDisableTiming));
        OFDM_CUDA(ctx, cudaEventCreateWithFlags(&ctx->call_start, cudaEventDisableTiming));
    }
    // Host->device copies (copy stream) are pipelined against the sweep of the previous chunk (compute stream):
    // chunk c's kernels wait only for chunk c's copies.  The scratch buffers may still be read by earlier work
    // on the compute stream, so the copy stream first waits for everything enqueued there so far.
    OFDM_CUDA(ctx, cudaEventRecord(ctx->call_start, ctx->stream));
    OFDM_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->call_start, 0));
    OFDM_CUDA(ctx, cudaMemsetAsync(cnt, 0, sizeof(ofdm_counters) * (size_t)n_snr, ctx->stream));
    const long chunk = 65536;
    int c = 0;
    for (long f0 = 0; f0 < n_frames; f0 += chunk, ++c) {
        const long n = n_frames - f0 < chunk ? n_frames - f0 : chunk;
        char *db = (char *)bits + f0 * bits_per_frame, *dg = (char *)g + f0 * g_per_frame;
        OFDM_CUDA(ctx, cudaMemcpyAsync(db, (const char *)bits_host + f0 * bits_per_frame, n * bits_per_frame, cudaMemcpyHostToDevice, ctx->copy_stream));
        const char *hg = (const char *)g_host + f0 * g_per_frame;
        if (n_sym <= 4) {
            // The receiver never reads the draws of the guard interval and the cyclic prefixes (Channel_Estimation :837-838
            // and the CP strip :1028 skip those samples), so they stay on the host: strided copies of the LTS halves and of
            // each symbol body -- 20 % fewer bytes over PCIe for the default frame.  The device buffer keeps the full layout.
            OFDM_CUDA(ctx, cudaMemcpy2DAsync(dg + 32 * 4, g_per_frame, hg + 32 * 4, g_per_frame, 128 * 4, n, cudaMemcpyHostToDevice, ctx->copy_stream));
            for (int sy = 0; sy < n_sym; ++sy) {
                const size_t off = (size_t)(160 + 80 * sy + 16) * 4;
                OFDM_CUDA(ctx, cudaMemcpy2DAsync(dg + off, g_per_frame, hg + off, g_per_frame, 64 * 4, n, cudaMemcpyHostToDevice, ctx->copy_stream));
            }
        } else {
            OFDM_CUDA(ctx, cudaMemcpyAsync(dg, hg, n * g_per_frame, cudaMemcpyHostToDevice, ctx->copy_stream));
        }
        OFDM_CUDA(ctx, cudaEventRecord(ctx->copy_done[c & 1], ctx->copy_stream));
        OFDM_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->copy_done[c & 1], 0));
        float *fr = (float *)frames + f0 * len * 2, *pw = (float *)power + f0;
        if (int st = ofdm_tx_frames(ctx, (const uint32_t *)db, fr, pw, n, n_sym, mode)) return st;        // Transmitter(), OFDM.c:1191
        if (int st = sweep_points(ctx, fr, (const float *)dg, pw, (const uint32_t *)db, n, n_sym, snr_db, n_snr, mode,     // SNR loop, OFDM.c:1202-1222
                                  (ofdm_counters *)cnt))
            return st;
    }
    OFDM_CUDA(ctx, cudaMemcpyAsync(out_host, cnt, sizeof(ofdm_counters) * (size_t)n_snr, cudaMemcpyDeviceToHost, ctx->stream));
    OFDM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return OFDM_OK;
}

}  // extern "C"

namespace {
int sweep_points(ofdm_ctx *ctx, const float *frames, const float *g, const float *power, const uint32_t *bits, long n_frames, int n_sym,
                 const float *snr_db, int n_snr, int mode, ofdm_counters *counters)
{
    const bool aligned = ((uintptr_t)frames % 16 == 0) && ((uintptr_t)g % 16 == 0);
    const bool fused = ctx->fused_sweep && n_sym == 2 && aligned && !ctx->force_generic && !ctx->general_stream &&
                       (mode != OFDM_MODE_EXACT || ctx->checked);
    if (!fused) {
        for (int i = 0; i < n_snr; ++i)
            if (int st = ofdm_awgn_rx_inject(ctx, frames, g, power, bits, snr_db[i], n_frames, n_sym, mode, counters + i, nullptr)) return st;
        return OFDM_OK;
    }
    const long max_frames = 1L << 30;                      // per launch: the per-lane totals are 32-bit
    for (int s0 = 0; s0 < n_snr; s0 += kMaxSnr) {
        SweepParams p;
        memset(&p, 0, sizeof p);
        p.n_snr = n_snr - s0 < kMaxSnr ? n_snr - s0 : kMaxSnr;
        for (int i = 0; i < p.n_snr; ++i) p.snr_lin[i] = snr_linear(snr_db[s0 + i]);
        p.radius_scale = ctx->force_replay ? INFINITY : kRadius;
        p.replayed = ctx->replayed_dev;
        p.evm_guard = ctx->evm_guard;
        p.counters = counters + s0;
        for (long f0 = 0; f0 < n_frames; f0 += max_frames) {
            p.n_frames = n_frames - f0 < max_frames ? n_frames - f0 : max_frames;
            p.in = reinterpret_cast<const float2 *>(frames) + f0 * 320;
            p.g = g + f0 * 320;
            p.power = power + f0;
            p.tx_bits = bits + f0 * 6;
            auto launch = [&](auto k) -> int {                          // the kernel's own block shape
                constexpr int warps = kSweepWarps;
                const size_t smem = sweep_smem_bytes(warps);
                OFDM_CUDA(ctx, allow_smem(ctx, k, smem));
                const int grid = grid_for(ctx, k, smem, warps, p.n_frames, warps * 32);            // a warp works on one frame at a time
                k<<<grid, warps * 32, smem, ctx->stream>>>(p);
                return check_launch(ctx, "k_sweep_lin");
            };
            if (int st = mode == OFDM_MODE_EXACT ? launch(k_sweep_lin<kArithChecked>) : launch(k_sweep_lin<kArithFast>)) return st;
        }
    }
    return OFDM_OK;
}
}  // namespace

extern "C" {

// ------------------------------------------------------------------ Philox Monte-Carlo
int ofdm_random_bits(ofdm_ctx *ctx, uint32_t seed, uint64_t frame0, long n_frames, int n_sym, uint32_t *bits)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym));
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, bits != nullptr);
    long n = n_frames * n_sym;
    k_philox_bits<<<blocks_1d(n), 256, 0, ctx->stream>>>(seed, frame0, n, n_sym, bits);
    return check_launch(ctx, "k_philox_bits");
}

}  // extern "C"

namespace {
// McParams of the sweep of one frame range over a list of points through channel ch; streams[i] (nullable: i) is the Philox
// noise stream of point i.  The noise scale inv_sqrt_snr is 1 / sqrt(snr) for the reference channel, sigma / sqrt(P) for the
// other frame-power ones and sigma itself for Es/N0 and Eb/N0 (kChFixedSigma), each in its own rounding.  Only the reference
// channel's kernels speculate (error radii, replay counter).
McParams mc_params(const ofdm_ctx *ctx, const ofdm_channel &ch, uint32_t seed, uint64_t frame0, long n_frames, const float *snr_db,
                   const uint32_t *streams, int n_snr, ofdm_counters *counters)
{
    const bool reference = is_reference_channel(ch.noise, ch.snr_def), fixed = ch.snr_def != OFDM_SNR_FRAME_POWER;
    const double rail_share = ch.noise == OFDM_NOISE_COMPLEX ? 0.5 : 1.0;      // complex noise: half of the noise power per rail
    McParams p;
    memset(&p, 0, sizeof p);
    p.seed = seed; p.frame0 = frame0; p.n_frames = n_frames;
    p.n_snr = n_snr; p.counters = counters; p.n_taps = ch.n_taps;
    for (int i = 0; i < n_snr; ++i) {
        if (fixed) p.inv_sqrt_snr[i] = (float)sqrt(rail_share * (double)fixed_noise_power(ch.snr_def, snr_db[i]));
        else {
            p.snr_lin[i] = snr_linear(snr_db[i]);
            p.inv_sqrt_snr[i] = reference ? (float)(1.0 / sqrt((double)p.snr_lin[i])) : (float)sqrt(rail_share / (double)p.snr_lin[i]);
        }
        p.stream[i] = streams ? streams[i] : (uint32_t)i;
    }
    if (reference) {
        p.radius_scale = ctx->force_replay ? INFINITY : kRadius;
        p.replayed = ctx->replayed_dev;
        p.evm_guard = ctx->evm_guard;
        p.radius_chan = ctx->force_replay ? INFINITY : kChanRadius * sqrtf(320.f) * 1.001f;
    }
    return p;
}

// fused Monte-Carlo sweep of two-symbol frames, everything on chip: k_mc_quad works on four frames per warp in blocks of
// kMcQuadWarps warps, k_mc_philox on one frame per warp.  One launch per 2^30 frames: the per-lane totals are 32-bit.
template <typename K>
int mc_fused(ofdm_ctx *ctx, K k, bool quad, const McParams &all)
{
    const bool mp = all.n_taps > 0;
    const size_t smem = quad ? (mp ? mc_quad_mp_smem_bytes() : mc_quad_smem_bytes()) : mc_smem_bytes(mp);
    const long max_frames = 1L << 30;
    for (long f0 = 0; f0 < all.n_frames; f0 += max_frames) {
        McParams p = all;
        p.frame0 = all.frame0 + (uint64_t)f0;
        p.n_frames = all.n_frames - f0 < max_frames ? all.n_frames - f0 : max_frames;
        const int st = quad ? launch_persistent(ctx, k, kMcQuadWarps, 4, smem, p, "k_mc_quad")
                            : launch_persistent(ctx, k, kWarpsPerBlock, 1, smem, p, "k_mc_philox");
        if (st) return st;
    }
    return OFDM_OK;
}

// staged Monte-Carlo sweep, frames in HBM per chunk of at most 2 GiB: Philox bits, transmitter, [taps, frame power of the faded
// frames], then per point the reference channel's fused channel + receiver (ofdm_awgn_rx_philox), or another channel
// (k_awgn_channel) into an OTA buffer and the verified receiver of ofdm_rx_frames on it.  Without taps the frame power comes
// from the transmitter (its LTS-prefix shortcut).
// With a code (nullable) the Philox bits are the information bits: k_conv_encode turns them into the payload the transmitter
// sends, the receiver dumps H and eq of every point (its own counters go to raw, nullable) and k_viterbi decodes them and counts
// the information-bit errors into counters.  Eb/N0 points then count information bits (fixed_noise_power).
int mc_staged(ofdm_ctx *ctx, const ofdm_channel &ch, const ofdm_code *code, uint32_t seed, uint64_t frame0, long n_frames, int n_sym,
              const float *snr_db, const uint32_t *streams, int n_snr, int mode, ofdm_counters *counters, ofdm_counters *raw)
{
    const int len = OFDM_FRAME_LEN(n_sym);
    const bool reference = is_reference_channel(ch.noise, ch.snr_def), per_frame = ch.snr_def == OFDM_SNR_FRAME_POWER, mp = ch.n_taps > 0;
    const long dump_bytes = code ? (64L + 48L * n_sym) * 8 : 0;       // H and eq of a frame
    long chunk = (2L << 30) / ((long)len * 8 + dump_bytes);
    if (chunk < 1024) chunk = 1024;
    for (long f0 = 0; f0 < n_frames; f0 += chunk) {
        const long n = n_frames - f0 < chunk ? n_frames - f0 : chunk;
        const size_t frame_bytes = (size_t)n * len * 2 * sizeof(float), word_bytes = (size_t)n * n_sym * 3 * sizeof(uint32_t);
        void *bits = nullptr, *frames = nullptr, *power = nullptr, *faded = nullptr, *ota = nullptr, *payload = nullptr;
        ofdm_rx_dump dump;
        memset(&dump, 0, sizeof dump);
        if (int st = ensure_scratch(ctx, 4, word_bytes, &bits)) return st;
        if (int st = ensure_scratch(ctx, 1, frame_bytes, &frames)) return st;
        if (mp) if (int st = ensure_scratch(ctx, 5, frame_bytes, &faded)) return st;
        if (!reference) if (int st = ensure_scratch(ctx, 6, frame_bytes, &ota)) return st;
        if (per_frame) if (int st = ensure_scratch(ctx, 2, (size_t)n * sizeof(float), &power)) return st;
        if (code) {
            void *H = nullptr, *eq = nullptr;
            if (int st = ensure_scratch(ctx, 7, word_bytes, &payload)) return st;
            if (int st = ensure_scratch(ctx, 8, (size_t)n * 64 * 2 * sizeof(float), &H)) return st;
            if (int st = ensure_scratch(ctx, 9, (size_t)n * n_sym * 48 * 2 * sizeof(float), &eq)) return st;
            dump.H = (float *)H;
            dump.eq = (float *)eq;
        }
        const uint64_t fr0 = frame0 + (uint64_t)f0;
        if (int st = ofdm_random_bits(ctx, seed, fr0, n, n_sym, (uint32_t *)bits)) return st;
        if (code) if (int st = launch_conv_encode(ctx, code->rate, (const uint32_t *)bits, (uint32_t *)payload, n, n_sym)) return st;
        const uint32_t *sent = (const uint32_t *)(code ? payload : bits);
        const ofdm_rx_dump *dp = code ? &dump : nullptr;
        if (int st = ofdm_tx_frames(ctx, sent, (float *)frames, mp ? nullptr : (float *)power, n, n_sym, mode)) return st;
        const float *air = (const float *)frames;
        if (mp) {
            if (int st = ofdm_multipath_philox(ctx, air, seed, fr0, ch.n_taps, (float *)faded, nullptr, n, n_sym)) return st;
            air = (const float *)faded;
            if (per_frame) if (int st = frame_power(ctx, air, (float *)power, n, len, mode)) return st;     // power of what goes on the air
        }
        for (int i = 0; i < n_snr; ++i) {
            const uint32_t stream = streams ? streams[i] : (uint32_t)i;
            ofdm_counters *rx_cnt = code ? (raw ? raw + i : nullptr) : counters + i;
            if (reference) {
                if (int st = ofdm_awgn_rx_philox(ctx, air, (const float *)power, sent, snr_db[i], seed, stream, fr0, n, n_sym, mode, rx_cnt, dp))
                    return st;
            } else {
                const int st = per_frame ? launch_awgn_channel(ctx, ch.noise, air, (const float *)power, snr_linear(snr_db[i]), 0.f, seed, stream,
                                                               fr0, (float *)ota, n, len, mode)
                                         : launch_awgn_channel(ctx, ch.noise, air, nullptr, 1.f,
                                                               fixed_noise_power(ch.snr_def, snr_db[i], info_bits_per_point(code)), seed, stream, fr0,
                                                               (float *)ota, n, len, mode);
                if (st) return st;
                if (int st2 = ofdm_rx_frames(ctx, (const float *)ota, sent, n, n_sym, mode, rx_cnt, dp)) return st2;
            }
            if (code)
                if (int st = launch_viterbi(ctx, *code, dump.H, dump.eq, (const uint32_t *)bits, nullptr, n, n_sym, counters + i)) return st;
        }
    }
    return OFDM_OK;
}

void add_counters(ofdm_counters &t, const ofdm_counters &q)
{
    t.bit_errors += q.bit_errors; t.bits += q.bits; t.frames_in_error += q.frames_in_error; t.rail_errors += q.rail_errors; t.frames += q.frames;
    t.sum_err2 += q.sum_err2; t.sum_ref2 += q.sum_ref2; t.sum_evm_lin += q.sum_evm_lin;
}

// The stop rule of configs[3]: rounds of round_frames frames (global indices frame0 + r * round_frames ...) until every point has
// >= target_errors bit errors or >= max_bits bits in out_host.  run_round(frame0, snr, streams, n_active, cnt, raw) accumulates
// one round of the still-active points into the zeroed device counters cnt [n_active] and, when raw_host is given, raw
// [n_active], which are summed into raw_host alongside.
template <typename R>
int until_rounds(ofdm_ctx *ctx, uint64_t frame0, const float *snr_db, int n_snr, uint64_t target_errors, uint64_t max_bits, long round_frames,
                 ofdm_counters *out_host, ofdm_counters *raw_host, int *rounds_out, R run_round)
{
    if (rounds_out) *rounds_out = 0;
    if (n_snr == 0) return OFDM_OK;
    memset(out_host, 0, sizeof(ofdm_counters) * (size_t)n_snr);
    if (raw_host) memset(raw_host, 0, sizeof(ofdm_counters) * (size_t)n_snr);
    void *buf = nullptr;
    if (int st = ensure_scratch(ctx, 3, sizeof(ofdm_counters) * 2 * (size_t)kMaxSnr, &buf)) return st;
    ofdm_counters *cnt = (ofdm_counters *)buf, *raw = raw_host ? cnt + kMaxSnr : nullptr;
    int active[kMaxSnr], n_active = n_snr, rounds = 0;
    for (int i = 0; i < n_snr; ++i) active[i] = i;
    ofdm_counters part[kMaxSnr], part_raw[kMaxSnr];
    while (n_active > 0) {
        float snr_a[kMaxSnr];
        uint32_t stream_a[kMaxSnr];
        for (int j = 0; j < n_active; ++j) { snr_a[j] = snr_db[active[j]]; stream_a[j] = (uint32_t)active[j]; }
        OFDM_CUDA(ctx, cudaMemsetAsync(cnt, 0, sizeof(ofdm_counters) * (size_t)(raw ? 2 * kMaxSnr : n_active), ctx->stream));
        if (int st = run_round(frame0 + (uint64_t)rounds * (uint64_t)round_frames, snr_a, stream_a, n_active, cnt, raw)) return st;
        OFDM_CUDA(ctx, cudaMemcpyAsync(part, cnt, sizeof(ofdm_counters) * (size_t)n_active, cudaMemcpyDeviceToHost, ctx->stream));
        if (raw) OFDM_CUDA(ctx, cudaMemcpyAsync(part_raw, raw, sizeof(ofdm_counters) * (size_t)n_active, cudaMemcpyDeviceToHost, ctx->stream));
        OFDM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        int keep = 0;
        for (int j = 0; j < n_active; ++j) {
            ofdm_counters &t = out_host[active[j]];
            add_counters(t, part[j]);
            if (raw) add_counters(raw_host[active[j]], part_raw[j]);
            if (t.bit_errors < target_errors && t.bits < max_bits) active[keep++] = active[j];   // the stop rule of configs[3]
        }
        n_active = keep;
        ++rounds;
    }
    if (rounds_out) *rounds_out = rounds;
    return OFDM_OK;
}
}  // namespace

extern "C" {

int ofdm_mc_sweep_philox_dev(ofdm_ctx *ctx, uint32_t seed, uint64_t frame0, long n_frames, int n_sym, const float *snr_db,
                             int n_snr, int mode, ofdm_counters *counters)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && mode_ok(mode) && n_snr >= 0 && n_snr <= kMaxSnr);
    if (n_frames == 0 || n_snr == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, snr_db != nullptr && counters != nullptr);
    const ofdm_channel ch = {OFDM_NOISE_REAL_RAIL, OFDM_SNR_FRAME_POWER, 0};
    return ofdm_mc_sweep_channel_dev(ctx, &ch, seed, frame0, n_frames, n_sym, snr_db, nullptr, n_snr, mode, counters);
}

int ofdm_mc_sweep_points_dev(ofdm_ctx *ctx, uint32_t seed, uint64_t frame0, long n_frames, int n_sym, int n_taps, const float *snr_db,
                             const uint32_t *streams, int n_points, int mode, ofdm_counters *counters)
{
    const ofdm_channel ch = {OFDM_NOISE_REAL_RAIL, OFDM_SNR_FRAME_POWER, n_taps};
    return ofdm_mc_sweep_channel_dev(ctx, &ch, seed, frame0, n_frames, n_sym, snr_db, streams, n_points, mode, counters);
}

int ofdm_mc_sweep_channel_dev(ofdm_ctx *ctx, const ofdm_channel *ch, uint32_t seed, uint64_t frame0, long n_frames, int n_sym,
                              const float *snr_db, const uint32_t *streams, int n_points, int mode, ofdm_counters *counters)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, ch != nullptr && noise_ok(ch->noise) && snr_def_ok(ch->snr_def) && ch->n_taps >= 0 && ch->n_taps <= kMaxTaps);
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && mode_ok(mode) && n_points >= 0 && n_points <= kMaxSnr);
    if (n_frames == 0 || n_points == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, snr_db != nullptr && counters != nullptr);
    // Fused on chip (two-symbol frames only) or staged through HBM.  The reference channel without taps always fuses two-symbol
    // frames.  With taps, "multipath_path" chooses (0 = auto); measured per 1 M frames x 21 SNR points: fast 14.8 ms fused vs
    // 16.9 ms staged, exact 27.3 ms fused vs 20.0 ms staged (the fused kernel runs each frame's exact power chain on one lane, the
    // staged path one chain per lane).  The other channels fuse only in fp32.
    const bool reference = is_reference_channel(ch->noise, ch->snr_def), mp = ch->n_taps > 0, fast = mode != OFDM_MODE_EXACT;
    bool fused = n_sym == 2;
    if (!reference) fused = fused && fast && !ctx->force_generic;
    else if (mp) fused = fused && !ctx->force_generic && (ctx->multipath_path == 2 || (ctx->multipath_path == 0 && fast));
    if (!fused) return mc_staged(ctx, *ch, nullptr, seed, frame0, n_frames, n_sym, snr_db, streams, n_points, mode, counters, nullptr);
    const McParams p = mc_params(ctx, *ch, seed, frame0, n_frames, snr_db, streams, n_points, counters);
    auto quad = [&](auto k) { return mc_fused(ctx, k, true, p); };
    if (!reference) {                   // k_mc_quad<fast, MP, CH>: the channel is a compile-time parameter
        constexpr int C = kChComplex, F = kChFixedSigma;
        const bool cx = ch->noise == OFDM_NOISE_COMPLEX, fixed = ch->snr_def != OFDM_SNR_FRAME_POWER;
        auto go = [&](auto m) -> int {
            constexpr bool M = decltype(m)::value;
            return cx ? (fixed ? quad(k_mc_quad<kArithFast, M, C | F>) : quad(k_mc_quad<kArithFast, M, C>)) : quad(k_mc_quad<kArithFast, M, F>);
        };
        return mp ? go(std::true_type()) : go(std::false_type());
    }
    // one frame per lane group (k_mc_quad, ofdm_mc_quad.cuh) for the speculating arithmetic without taps and for fp32 with taps;
    // "stream_layout" = 1 and the all-exact arithmetic keep the one-frame-per-warp kernel
    return with_arith(arith_of(ctx, mode), [&](auto a) -> int {
        constexpr int A = decltype(a)::value;
        if constexpr (A == kArithFast) {
            if (ctx->stream_layout == 0) return mp ? quad(k_mc_quad<A, true>) : quad(k_mc_quad<A>);
        }
        if constexpr (A == kArithChecked) {
            if (ctx->stream_layout == 0 && !mp) return quad(k_mc_quad<A>);
        }
        return mp ? mc_fused(ctx, k_mc_philox<A, true>, false, p) : mc_fused(ctx, k_mc_philox<A>, false, p);
    });
}

int ofdm_mc_sweep_until(ofdm_ctx *ctx, uint32_t seed, uint64_t frame0, int n_sym, int n_taps, const float *snr_db, int n_snr, int mode,
                        uint64_t target_errors, uint64_t max_bits, long round_frames, ofdm_counters *out_host, int *rounds_out)
{
    const ofdm_channel ch = {OFDM_NOISE_REAL_RAIL, OFDM_SNR_FRAME_POWER, n_taps};
    return ofdm_mc_sweep_channel_until(ctx, &ch, seed, frame0, n_sym, snr_db, n_snr, mode, target_errors, max_bits, round_frames, out_host,
                                       rounds_out);
}

int ofdm_mc_sweep_channel_until(ofdm_ctx *ctx, const ofdm_channel *ch, uint32_t seed, uint64_t frame0, int n_sym, const float *snr_db,
                                int n_snr, int mode, uint64_t target_errors, uint64_t max_bits, long round_frames, ofdm_counters *out_host,
                                int *rounds_out)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, ch != nullptr && noise_ok(ch->noise) && snr_def_ok(ch->snr_def) && ch->n_taps >= 0 && ch->n_taps <= kMaxTaps);
    OFDM_REQUIRE(ctx, nsym_ok(n_sym) && mode_ok(mode) && n_snr >= 0 && n_snr <= kMaxSnr);
    OFDM_REQUIRE(ctx, round_frames >= 1 && max_bits >= 1 && (n_snr == 0 || (snr_db != nullptr && out_host != nullptr)));
    return until_rounds(ctx, frame0, snr_db, n_snr, target_errors, max_bits, round_frames, out_host, nullptr, rounds_out,
                        [&](uint64_t fr0, const float *snr, const uint32_t *streams, int n_points, ofdm_counters *cnt, ofdm_counters *) {
                            return ofdm_mc_sweep_channel_dev(ctx, ch, seed, fr0, round_frames, n_sym, snr, streams, n_points, mode, cnt);
                        });
}

// ------------------------------------------------------------------ the coded link (DESIGN.md section 6.2)
int ofdm_conv_encode(ofdm_ctx *ctx, int rate, const uint32_t *info, uint32_t *payload, long n_frames, int n_sym)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, rate_ok(rate) && n_frames >= 0 && nsym_ok(n_sym));
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, info != nullptr && payload != nullptr && (const void *)info != (const void *)payload);
    return launch_conv_encode(ctx, rate, info, payload, n_frames, n_sym);
}

int ofdm_viterbi_decode(ofdm_ctx *ctx, const ofdm_code *code, const float *H, const float *eq, const uint32_t *info, uint32_t *decoded,
                        long n_frames, int n_sym, ofdm_counters *counters)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, code_ok(code) && n_frames >= 0 && nsym_ok(n_sym));
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, H != nullptr && eq != nullptr && (counters == nullptr || info != nullptr));
    return launch_viterbi(ctx, *code, H, eq, info, decoded, n_frames, n_sym, counters);
}

int ofdm_mc_sweep_coded_dev(ofdm_ctx *ctx, const ofdm_channel *ch, const ofdm_code *code, uint32_t seed, uint64_t frame0, long n_frames,
                            int n_sym, const float *snr_db, const uint32_t *streams, int n_points, int mode, ofdm_counters *coded,
                            ofdm_counters *raw)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, ch != nullptr && noise_ok(ch->noise) && snr_def_ok(ch->snr_def) && ch->n_taps >= 0 && ch->n_taps <= kMaxTaps);
    OFDM_REQUIRE(ctx, code_ok(code));
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && mode_ok(mode) && n_points >= 0 && n_points <= kMaxSnr);
    if (n_frames == 0 || n_points == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, snr_db != nullptr && coded != nullptr);
    return mc_staged(ctx, *ch, code, seed, frame0, n_frames, n_sym, snr_db, streams, n_points, mode, coded, raw);
}

int ofdm_mc_sweep_coded_until(ofdm_ctx *ctx, const ofdm_channel *ch, const ofdm_code *code, uint32_t seed, uint64_t frame0, int n_sym,
                              const float *snr_db, int n_snr, int mode, uint64_t target_errors, uint64_t max_bits, long round_frames,
                              ofdm_counters *coded_host, ofdm_counters *raw_host, int *rounds_out)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, ch != nullptr && noise_ok(ch->noise) && snr_def_ok(ch->snr_def) && ch->n_taps >= 0 && ch->n_taps <= kMaxTaps);
    OFDM_REQUIRE(ctx, code_ok(code));
    OFDM_REQUIRE(ctx, nsym_ok(n_sym) && mode_ok(mode) && n_snr >= 0 && n_snr <= kMaxSnr);
    OFDM_REQUIRE(ctx, round_frames >= 1 && max_bits >= 1 && (n_snr == 0 || (snr_db != nullptr && coded_host != nullptr)));
    return until_rounds(ctx, frame0, snr_db, n_snr, target_errors, max_bits, round_frames, coded_host, raw_host, rounds_out,
                        [&](uint64_t fr0, const float *snr, const uint32_t *streams, int n_points, ofdm_counters *cnt, ofdm_counters *raw) {
                            return ofdm_mc_sweep_coded_dev(ctx, ch, code, seed, fr0, round_frames, n_sym, snr, streams, n_points, mode, cnt, raw);
                        });
}

int ofdm_mc_sweep_philox(ofdm_ctx *ctx, uint32_t seed, uint64_t frame0, long n_frames, int n_sym, const float *snr_db,
                         int n_snr, int mode, ofdm_counters *out_host)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_snr >= 0 && n_snr <= kMaxSnr && (n_snr == 0 || out_host != nullptr));
    if (n_snr > 0) memset(out_host, 0, sizeof(ofdm_counters) * (size_t)n_snr);
    if (n_snr == 0 || n_frames == 0) return OFDM_OK;
    void *cnt = nullptr;
    if (int st = ensure_scratch(ctx, 3, sizeof(ofdm_counters) * (size_t)n_snr, &cnt)) return st;
    OFDM_CUDA(ctx, cudaMemsetAsync(cnt, 0, sizeof(ofdm_counters) * (size_t)n_snr, ctx->stream));
    if (int st = ofdm_mc_sweep_philox_dev(ctx, seed, frame0, n_frames, n_sym, snr_db, n_snr, mode, (ofdm_counters *)cnt)) return st;
    OFDM_CUDA(ctx, cudaMemcpyAsync(out_host, cnt, sizeof(ofdm_counters) * (size_t)n_snr, cudaMemcpyDeviceToHost, ctx->stream));
    OFDM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return OFDM_OK;
}

// ------------------------------------------------------------------ multipath extension (configs[4])
static int multipath_common(ofdm_ctx *ctx, bool philox, const float *tx, const float *taps, uint32_t seed, uint64_t frame0, int n_taps,
                            float *out, float *taps_out, long n_frames, int n_sym)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && n_taps >= 1 && n_taps <= kMaxTaps);
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, tx != nullptr && out != nullptr && tx != out && (philox || taps != nullptr));
    const int len = OFDM_FRAME_LEN(n_sym);
    const int tile = fir_tile(len);
    const size_t smem = fir_smem_bytes(tile);
    const float2 *x = reinterpret_cast<const float2 *>(tx), *h = reinterpret_cast<const float2 *>(taps);
    float2 *y = reinterpret_cast<float2 *>(out), *ho = reinterpret_cast<float2 *>(taps_out);
    if (philox) {
        if (smem > 48 * 1024) OFDM_CUDA(ctx, allow_smem(ctx, k_multipath<true>, fir_smem_bytes(kFirTile)));
        int grid = grid_for(ctx, k_multipath<true>, smem, kWarpsPerBlock, n_frames);
        k_multipath<true><<<grid, kThreads, smem, ctx->stream>>>(x, h, seed, frame0, n_taps, y, ho, n_frames, len, tile);
    } else {
        if (smem > 48 * 1024) OFDM_CUDA(ctx, allow_smem(ctx, k_multipath<false>, fir_smem_bytes(kFirTile)));
        int grid = grid_for(ctx, k_multipath<false>, smem, kWarpsPerBlock, n_frames);
        k_multipath<false><<<grid, kThreads, smem, ctx->stream>>>(x, h, seed, frame0, n_taps, y, ho, n_frames, len, tile);
    }
    return check_launch(ctx, "k_multipath");
}

int ofdm_multipath_taps(ofdm_ctx *ctx, const float *tx, const float *taps, int n_taps, float *out, long n_frames, int n_sym)
{
    return multipath_common(ctx, false, tx, taps, 0, 0, n_taps, out, nullptr, n_frames, n_sym);
}
int ofdm_multipath_philox(ofdm_ctx *ctx, const float *tx, uint32_t seed, uint64_t frame0, int n_taps, float *out, float *taps_out,
                          long n_frames, int n_sym)
{
    return multipath_common(ctx, true, tx, nullptr, seed, frame0, n_taps, out, taps_out, n_frames, n_sym);
}

int ofdm_mc_sweep_multipath_dev(ofdm_ctx *ctx, uint32_t seed, uint64_t frame0, long n_frames, int n_sym, int n_taps, const float *snr_db,
                                int n_snr, int mode, ofdm_counters *counters)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && nsym_ok(n_sym) && mode_ok(mode) && n_snr >= 0 && n_snr <= kMaxSnr && n_taps >= 1 && n_taps <= kMaxTaps);
    if (n_frames == 0 || n_snr == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, snr_db != nullptr && counters != nullptr);
    const ofdm_channel ch = {OFDM_NOISE_REAL_RAIL, OFDM_SNR_FRAME_POWER, n_taps};
    return ofdm_mc_sweep_channel_dev(ctx, &ch, seed, frame0, n_frames, n_sym, snr_db, nullptr, n_snr, mode, counters);
}


// ------------------------------------------------------------------ pulse shaping (SURVEY 8(f) rank 1)
int ofdm_rrc_tx(ofdm_ctx *ctx, const float *frames, float *out, long n_frames, int frame_len)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && frame_len >= 1 && frame_len <= OFDM_FRAME_LEN(OFDM_MAX_SYM));
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, frames != nullptr && out != nullptr && frames != out);
    const int tile = fir_tile(frame_len);
    const size_t smem = fir_smem_bytes(tile);
    if (smem > 48 * 1024) OFDM_CUDA(ctx, allow_smem(ctx, k_rrc_tx, fir_smem_bytes(kFirTile)));
    int grid = grid_for(ctx, k_rrc_tx, smem, kWarpsPerBlock, n_frames);
    k_rrc_tx<<<grid, kThreads, smem, ctx->stream>>>(reinterpret_cast<const float2 *>(frames), reinterpret_cast<float2 *>(out), n_frames, frame_len, tile);
    return check_launch(ctx, "k_rrc_tx");
}
int ofdm_rrc_rx(ofdm_ctx *ctx, const float *in, float *out, long n_frames, int in_len, int packet_idx, int frame_len)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && in_len >= 1 && in_len <= 2 * OFDM_FRAME_LEN(OFDM_MAX_SYM) + 64 && frame_len >= 1 && packet_idx >= 0);
    // the reference reads Rx_filter_signal[packet_idx + 2*(frame_len-1)] (:992-994): it must exist (in_len + 20 filtered samples)
    OFDM_REQUIRE(ctx, (long)packet_idx + 2L * (frame_len - 1) < (long)in_len + 20);
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, in != nullptr && out != nullptr && in != out);
    const int tile = fir_tile(2 * frame_len);
    const size_t smem = fir_smem_bytes(tile);
    if (smem > 48 * 1024) OFDM_CUDA(ctx, allow_smem(ctx, k_rrc_rx, fir_smem_bytes(kFirTile)));
    int grid = grid_for(ctx, k_rrc_rx, smem, kWarpsPerBlock, n_frames);
    k_rrc_rx<<<grid, kThreads, smem, ctx->stream>>>(reinterpret_cast<const float2 *>(in), nullptr, packet_idx, reinterpret_cast<float2 *>(out), n_frames,
                                                   in_len, frame_len, tile);
    return check_launch(ctx, "k_rrc_rx");
}
int ofdm_awgn_inject_len(ofdm_ctx *ctx, const float *tx, const float *g, const float *power, float snr_db, float *ota, long n_frames,
                         int frame_len, int mode)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && frame_len >= 1 && frame_len <= (1 << 24) && mode_ok(mode));
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, tx != nullptr && ota != nullptr && g != nullptr);
    const float *pw = nullptr;
    if (int st = resolve_power(ctx, tx, power, n_frames, frame_len, mode, &pw)) return st;
    const float2 *x = reinterpret_cast<const float2 *>(tx);
    float2 *y = reinterpret_cast<float2 *>(ota);
    const float sl = snr_linear(snr_db);
    if (mode == OFDM_MODE_EXACT) {
        int grid = grid_for(ctx, k_awgn<true, kNoiseInject>, 0, kWarpsPerBlock, n_frames);
        k_awgn<true, kNoiseInject><<<grid, kThreads, 0, ctx->stream>>>(x, g, pw, sl, 0, 0, 0, y, n_frames, frame_len);
    } else {
        int grid = grid_for(ctx, k_awgn<false, kNoiseInject>, 0, kWarpsPerBlock, n_frames);
        k_awgn<false, kNoiseInject><<<grid, kThreads, 0, ctx->stream>>>(x, g, pw, sl, 0, 0, 0, y, n_frames, frame_len);
    }
    return check_launch(ctx, "k_awgn");
}

// ------------------------------------------------------------------ packet detection / selection (SURVEY 8(f) rank 2)
int ofdm_packet_detect(ofdm_ctx *ctx, const float *rx, float *corr, long n, int len)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n >= 0 && len >= 48);
    if (n == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, rx != nullptr && corr != nullptr);
    int tile = (len - 47 + 31) & ~31;
    if (tile > 4096) tile = 4096;
    const size_t smem = (size_t)(tile + 48) * (sizeof(double) + sizeof(float2));
    if (smem > 48 * 1024) OFDM_CUDA(ctx, allow_smem(ctx, k_packet_detect, ((4096 + 48) * 16)));
    int grid = grid_for(ctx, k_packet_detect, smem, 1, n);                  // one capture per block iteration, all resident blocks
    k_packet_detect<<<grid, kThreads, smem, ctx->stream>>>(reinterpret_cast<const float2 *>(rx), corr, n, len, tile);
    return check_launch(ctx, "k_packet_detect");
}
int ofdm_packet_select(ofdm_ctx *ctx, const float *corr, int32_t *idx, long n, int len_corr)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n >= 0 && len_corr >= 1);
    if (n == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, corr != nullptr && idx != nullptr);
    int grid = grid_for(ctx, k_packet_select, 0, kWarpsPerBlock, n);
    k_packet_select<<<grid, kThreads, 0, ctx->stream>>>(corr, idx, n, len_corr);
    return check_launch(ctx, "k_packet_select");
}

// ------------------------------------------------------------------ CFO and full-path glue (SURVEY 8(f) ranks 3, 4)
int ofdm_sts(ofdm_ctx *ctx, float *sts_time_host)
{
    if (!ctx || !sts_time_host) return OFDM_ERR_INVALID;
    memcpy(sts_time_host, ctx->sts_time, sizeof ctx->sts_time);
    return OFDM_OK;
}
int ofdm_prepend_sts(ofdm_ctx *ctx, const float *frames, float *out, long n_frames, int frame_len)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && frame_len >= 1);
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, frames != nullptr && out != nullptr && frames != out);
    long total = n_frames * (160 + (long)frame_len);
    int grid = (int)((total + 255) / 256 < 4L * ctx->sm_count * 8 ? (total + 255) / 256 : 4L * ctx->sm_count * 8);
    k_prepend<<<grid, 256, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(ctx->sts_dev), 160, reinterpret_cast<const float2 *>(frames),
                                             reinterpret_cast<float2 *>(out), n_frames, frame_len);
    return check_launch(ctx, "k_prepend");
}
int ofdm_gather(ofdm_ctx *ctx, const float *in, const int32_t *start, int start_scalar, float *out, long n, int in_len, int out_len)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n >= 0 && in_len >= 1 && out_len >= 1 && (start != nullptr || start_scalar >= 0));
    if (n == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, in != nullptr && out != nullptr && in != out);
    int grid = grid_for(ctx, k_gather, 0, kWarpsPerBlock, n);
    k_gather<<<grid, kThreads, 0, ctx->stream>>>(reinterpret_cast<const float2 *>(in), start, start_scalar, reinterpret_cast<float2 *>(out), n, in_len, out_len);
    return check_launch(ctx, "k_gather");
}
int ofdm_rrc_rx_idx(ofdm_ctx *ctx, const float *in, const int32_t *idx, float *out, long n_frames, int in_len, int frame_len)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && in_len >= 1 && frame_len >= 1);
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, in != nullptr && out != nullptr && idx != nullptr && in != out);
    const int tile = fir_tile(2 * frame_len);
    const size_t smem = fir_smem_bytes(tile);
    if (smem > 48 * 1024) OFDM_CUDA(ctx, allow_smem(ctx, k_rrc_rx, fir_smem_bytes(kFirTile)));
    int grid = grid_for(ctx, k_rrc_rx, smem, kWarpsPerBlock, n_frames);
    k_rrc_rx<<<grid, kThreads, smem, ctx->stream>>>(reinterpret_cast<const float2 *>(in), idx, 0, reinterpret_cast<float2 *>(out), n_frames, in_len, frame_len, tile);
    return check_launch(ctx, "k_rrc_rx(idx)");
}
static int cfo_common(ofdm_ctx *ctx, bool fine, const float *rx, float *out, float *freq, long n, int len)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n >= 0 && len >= (fine ? 320 : 112));
    if (n == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, rx != nullptr && out != nullptr && rx != out);
    const float2 *x = reinterpret_cast<const float2 *>(rx);
    float2 *y = reinterpret_cast<float2 *>(out);
    if (fine) {
        int grid = grid_for(ctx, k_cfo<true>, 0, kWarpsPerBlock, n);
        k_cfo<true><<<grid, kThreads, 0, ctx->stream>>>(x, y, freq, n, len);
    } else {
        int grid = grid_for(ctx, k_cfo<false>, 0, kWarpsPerBlock, n);
        k_cfo<false><<<grid, kThreads, 0, ctx->stream>>>(x, y, freq, n, len);
    }
    return check_launch(ctx, "k_cfo");
}
int ofdm_cfo_coarse(ofdm_ctx *ctx, const float *rx, float *out, float *freq, long n, int len) { return cfo_common(ctx, false, rx, out, freq, n, len); }
int ofdm_cfo_fine(ofdm_ctx *ctx, const float *rx, float *out, float *freq, long n, int len) { return cfo_common(ctx, true, rx, out, freq, n, len); }

int ofdm_awgn_philox_len(ofdm_ctx *ctx, const float *tx, const float *power, float snr_db, uint32_t seed, uint32_t stream, uint64_t frame0,
                         float *ota, long n_frames, int frame_len, int mode)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n_frames >= 0 && frame_len >= 1 && frame_len <= (1 << 24) && mode_ok(mode));
    if (n_frames == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, tx != nullptr && ota != nullptr);
    const float *pw = nullptr;
    if (int st = resolve_power(ctx, tx, power, n_frames, frame_len, mode, &pw)) return st;
    const float2 *x = reinterpret_cast<const float2 *>(tx);
    float2 *y = reinterpret_cast<float2 *>(ota);
    const float sl = snr_linear(snr_db);
    if (mode == OFDM_MODE_EXACT) {
        int grid = grid_for(ctx, k_awgn_philox_flat<true>, 0, kWarpsPerBlock, n_frames);
        k_awgn_philox_flat<true><<<grid, kThreads, 0, ctx->stream>>>(x, pw, sl, seed, stream, frame0, y, n_frames, frame_len);
    } else {
        int grid = grid_for(ctx, k_awgn_philox_flat<false>, 0, kWarpsPerBlock, n_frames);
        k_awgn_philox_flat<false><<<grid, kThreads, 0, ctx->stream>>>(x, pw, sl, seed, stream, frame0, y, n_frames, frame_len);
    }
    return check_launch(ctx, "k_awgn_philox_flat");
}

int ofdm_counters_pack(ofdm_ctx *ctx, const ofdm_counters *counters, int n, uint64_t *ints, double *dbls)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n >= 0);
    if (n == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, counters != nullptr && ints != nullptr && dbls != nullptr);
    k_counters_pack<<<blocks_1d(n), 256, 0, ctx->stream>>>(counters, n, reinterpret_cast<unsigned long long *>(ints), dbls);
    return check_launch(ctx, "k_counters_pack");
}
int ofdm_counters_unpack(ofdm_ctx *ctx, ofdm_counters *counters, int n, const uint64_t *ints, const double *dbls)
{
    if (int st = bind(ctx)) return st;
    OFDM_REQUIRE(ctx, n >= 0);
    if (n == 0) return OFDM_OK;
    OFDM_REQUIRE(ctx, counters != nullptr && ints != nullptr && dbls != nullptr);
    k_counters_unpack<<<blocks_1d(n), 256, 0, ctx->stream>>>(counters, n, reinterpret_cast<const unsigned long long *>(ints), dbls);
    return check_launch(ctx, "k_counters_unpack");
}

int ofdm_counters_finalize(const ofdm_counters *c, float res[3])
{
    if (!c || !res) return OFDM_ERR_INVALID;
    // evm = sqrt(err/N) / sqrt(ref/N), dB = 20*log10   OFDM.c:1124-1126; after the slicer every rail error
    // contributes (2/sqrt(2))^2 to the error energy, OFDM.c:1138-1139
    const double q = (double)kQpsk;
    double evm = sqrt(c->sum_err2 / c->sum_ref2);
    double evm_agc = sqrt((double)c->rail_errors * (2.0 * q) * (2.0 * q) / c->sum_ref2);
    res[0] = (float)(20.0 * log10(evm));
    res[1] = (float)(20.0 * log10(evm_agc));
    res[2] = c->bits ? (float)((double)c->bit_errors / (double)c->bits) : 0.f;   // OFDM.c:1161
    return OFDM_OK;
}

}  // extern "C"
