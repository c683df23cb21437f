"""The channels of ofdm_channel on the GPU (include/ofdm_b200.h, DESIGN.md "Channels"): the reference channel runs today's code,
the stage kernel and the EXACT sweeps match the channel oracle bit for bit on the GPU's own draws, the fused FAST sweep agrees
with the staged routes, results do not depend on how frames and points are split, and the complex / Es/N0 curve has the
statistics of an independent model."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from channel_oracle import ChannelOracle, model_complex_esn0

pytestmark = pytest.mark.gpu

SEED = 31
CHANNELS = [("complex", "frame_power"), ("complex", "esn0"), ("complex", "ebn0"), ("real", "esn0"), ("real", "ebn0")]
# the Es/N0 point whose noise power is exactly 2.0f: complex noise then has sigma = sqrt(0.5 * 2) = 1, and the channel on
# all-zero frames hands out the GPU's own normals bit for bit (no float32 SNR gives the real rail's sigma = 1 exactly)
SNR_UNIT_COMPLEX = -21.072099685668945


def ints(c):
    return (int(c.bit_errors), int(c.bits), int(c.frames_in_error), int(c.rail_errors), int(c.frames))


@pytest.fixture(scope="module")
def co():
    return ChannelOracle()


def gpu_draws(ofdm, pkg, stream, frame0, n_frames, n_sym):
    """the GPU's domain-0 and domain-4 normals of (SEED, stream) for frames [frame0, frame0 + n_frames), bit for bit"""
    assert np.float32(1.0 / (64.0 * 10.0 ** (SNR_UNIT_COMPLEX / 10.0))) == 2.0          # fixed_noise_power's arithmetic
    zeros = ofdm.zeros((n_frames, pkg.frame_len(n_sym), 2), ofdm.torch.float32)
    c = ofdm.awgn_philox_ex(zeros, SNR_UNIT_COMPLEX, SEED, stream, frame0, n_sym, pkg.MODE_EXACT, "complex", "esn0").cpu().numpy()
    return c[..., 0].copy(), c[..., 1].copy()


def test_draws_match_the_oracles_streams(ofdm, pkg, co):
    g0, g1 = gpu_draws(ofdm, pkg, 5, 12345678901, 64, 2)
    assert np.max(np.abs(g0 - co.philox_normals(SEED, 5, 12345678901, 64, 320, 0))) < 2e-5     # MUFU vs libm
    assert np.max(np.abs(g1 - co.philox_normals(SEED, 5, 12345678901, 64, 320, 4))) < 2e-5
    assert abs(g1.std() - 1) < 0.02 and abs(np.corrcoef(g0.ravel(), g1.ravel())[0, 1]) < 0.03


# ---- 1. the reference channel is today's code
@pytest.mark.parametrize("n_taps", [0, 4])
def test_reference_channel_is_todays_code(ofdm, pkg, n_taps):
    snrs = [0.0, 4.0, 9.0]
    for mode in (pkg.MODE_EXACT, pkg.MODE_FAST):
        a = ofdm.mc_sweep_channel(SEED, 100, 3001, 2, snrs, mode, n_taps=n_taps)
        cnt = ofdm.new_counters(3)
        ofdm.mc_sweep_points(SEED, 100, 3001, 2, n_taps, snrs, None, mode, cnt)
        b = ofdm.read_counters(cnt)
        assert [ints(x) for x in a] == [ints(x) for x in b]
        for x, y in zip(a, b):
            assert abs(x.sum_err2 - y.sum_err2) <= 1e-9 * y.sum_err2 and abs(x.sum_evm_lin - y.sum_evm_lin) <= 1e-9 * y.sum_evm_lin
        u1, r1 = ofdm.mc_sweep_channel_until(SEED, 0, 2, snrs, mode, n_taps=n_taps, target_errors=200, max_bits=3 * 2048 * 192,
                                             round_frames=2048)
        u2, r2 = ofdm.mc_sweep_until(SEED, 0, 2, n_taps, snrs, mode, 200, 3 * 2048 * 192, 2048)
        assert r1 == r2 and [ints(x) for x in u1] == [ints(x) for x in u2]
    bits = ofdm.random_bits(SEED, 9, 200, 3)
    tx, power = ofdm.tx_frames(bits, 3, pkg.MODE_EXACT)
    for mode in (pkg.MODE_EXACT, pkg.MODE_FAST):
        want = ofdm.awgn_philox(tx, 7.0, SEED, 2, 9, 3, mode)
        got = ofdm.awgn_philox_ex(tx, 7.0, SEED, 2, 9, 3, mode, "real", "frame_power")
        assert ofdm.torch.equal(want, got)


# ---- 2. the stage kernel
@pytest.mark.parametrize("n_sym", [1, 2, 5])
@pytest.mark.parametrize("noise,snr_def", CHANNELS)
def test_stage_kernel_against_oracle(ofdm, pkg, co, noise, snr_def, n_sym):
    n, frame0, stream = 37, 4000, 6
    bits = co.philox_bits(SEED, frame0, n, n_sym)
    tx, power = ofdm.tx_frames(ofdm.to_dev(pkg.pack_bits_host(bits).view(np.int32).reshape(-1)), n_sym, pkg.MODE_EXACT)
    tx_h = tx.cpu().numpy()
    g0, g1 = gpu_draws(ofdm, pkg, stream, frame0, n, n_sym)
    for snr in (-2.0, 7.5, 19.0):
        want = co.awgn_channel(tx_h, g0, g1 if noise == "complex" else None, snr, noise, snr_def)
        exact = ofdm.awgn_philox_ex(tx, snr, SEED, stream, frame0, n_sym, pkg.MODE_EXACT, noise, snr_def).cpu().numpy()
        assert np.array_equal(exact, want), (noise, snr_def, n_sym, snr)
        if snr_def == "frame_power":           # the supplied power gives the same bits as the internally computed one
            again = ofdm.awgn_philox_ex(tx, snr, SEED, stream, frame0, n_sym, pkg.MODE_EXACT, noise, snr_def, power=power).cpu().numpy()
            assert np.array_equal(again, want)
        fast = ofdm.awgn_philox_ex(tx, snr, SEED, stream, frame0, n_sym, pkg.MODE_FAST, noise, snr_def).cpu().numpy()
        # fp32 sigma and fmaf; the frame-power definition also sums the power in fp32 (another order than the reference's)
        tol = 1e-5 if snr_def == "frame_power" else 1e-6
        assert np.max(np.abs(fast - want)) <= tol * np.max(np.abs(want)), (noise, snr_def, n_sym, snr)


# ---- 3. EXACT sweeps against the oracle
def oracle_sweep(ofdm, pkg, co, frame0, n, n_sym, snrs, noise, snr_def, n_taps, streams=None):
    bits = co.philox_bits(SEED, frame0, n, n_sym)
    taps = None
    if n_taps > 0:
        tx = ofdm.tx_frames(ofdm.to_dev(pkg.pack_bits_host(bits).view(np.int32).reshape(-1)), n_sym, pkg.MODE_EXACT, with_power=False)
        taps = ofdm.multipath_philox(tx, SEED, frame0, n_taps, n_sym)[1].cpu().numpy()          # the GPU's own taps
    out = []
    for i, s in enumerate(snrs):
        g0, g1 = gpu_draws(ofdm, pkg, i if streams is None else streams[i], frame0, n, n_sym)
        out.append(co.chain_channel(bits, g0, g1 if noise == "complex" else None, taps, n_sym, s, noise, snr_def))
    return out


def assert_matches_oracle(got, want, what):
    for g, w in zip(got, want):
        assert ints(g) == ints(w), (what, ints(g), ints(w))
        assert abs(g.sum_err2 - w.sum_err2) <= 1e-5 * w.sum_err2, what
        assert abs(g.sum_evm_lin - w.sum_evm_lin) <= 1e-5 * w.sum_evm_lin, what


@pytest.mark.parametrize("n_taps", [0, 4])
@pytest.mark.parametrize("n_sym", [1, 2, 3])
@pytest.mark.parametrize("noise,snr_def", CHANNELS)
def test_exact_sweep_against_oracle(ofdm, pkg, co, noise, snr_def, n_sym, n_taps):
    n, frame0, snrs = 301, 777, [-1.0, 4.0, 9.0]
    want = oracle_sweep(ofdm, pkg, co, frame0, n, n_sym, snrs, noise, snr_def, n_taps)
    got = ofdm.mc_sweep_channel(SEED, frame0, n, n_sym, snrs, pkg.MODE_EXACT, noise, snr_def, n_taps)
    assert_matches_oracle(got, want, (noise, snr_def, n_sym, n_taps))
    if n_sym == 2:
        for opt, val, default in (("exact_speculation", 0, 1), ("force_replay", 1, 0)):
            ofdm.set_option(opt, val)
            try:
                again = ofdm.mc_sweep_channel(SEED, frame0, n, n_sym, snrs, pkg.MODE_EXACT, noise, snr_def, n_taps)
            finally:
                ofdm.set_option(opt, default)
            assert_matches_oracle(again, want, (opt, noise, snr_def, n_taps))


# ---- 4. FAST fused against the staged routes (same draws)
@pytest.mark.parametrize("n_taps", [0, 4])
@pytest.mark.parametrize("noise,snr_def", CHANNELS)
def test_fast_fused_against_staged(ofdm, pkg, noise, snr_def, n_taps):
    n, snrs = 3000, [0.0, 4.0, 8.0]
    fused = ofdm.mc_sweep_channel(SEED, 50, n, 2, snrs, pkg.MODE_FAST, noise, snr_def, n_taps)
    exact = ofdm.mc_sweep_channel(SEED, 50, n, 2, snrs, pkg.MODE_EXACT, noise, snr_def, n_taps)
    ofdm.set_option("force_generic_rx", 1)
    try:
        staged = ofdm.mc_sweep_channel(SEED, 50, n, 2, snrs, pkg.MODE_FAST, noise, snr_def, n_taps)
    finally:
        ofdm.set_option("force_generic_rx", 0)
    for other in (exact, staged):
        for a, b in zip(fused, other):
            assert (a.bits, a.frames) == (b.bits, b.frames)
            assert abs(a.bit_errors - b.bit_errors) <= 2 + 1e-5 * b.bit_errors and abs(a.rail_errors - b.rail_errors) <= 2 + 1e-5 * b.rail_errors
            assert abs(a.frames_in_error - b.frames_in_error) <= 2
            assert abs(a.sum_err2 - b.sum_err2) <= 5e-4 * b.sum_err2, (noise, snr_def, n_taps)


# ---- 5. split invariance and the until rule over ranks
@pytest.mark.parametrize("n_sym", [2, 3])
def test_split_invariance(ofdm, pkg, n_sym):
    snrs = [1.0, 5.0, 9.0]
    for noise, snr_def in (("complex", "esn0"), ("complex", "frame_power")):
        whole = ofdm.mc_sweep_channel(SEED, 1000, 1000, n_sym, snrs, pkg.MODE_EXACT, noise, snr_def)
        parts = [ofdm.mc_sweep_channel(SEED, 1000 + off, k, n_sym, snrs, pkg.MODE_EXACT, noise, snr_def) for off, k in ((0, 300), (300, 450), (750, 250))]
        for i in range(len(snrs)):
            assert tuple(sum(ints(p[i])[k] for p in parts) for k in range(5)) == ints(whole[i])
        last = ofdm.mc_sweep_channel(SEED, 1000, 1000, n_sym, snrs[2:], pkg.MODE_EXACT, noise, snr_def, streams=[2])
        assert ints(last[0]) == ints(whole[2])


def test_until_rule_over_ranks(ofdm, pkg):
    snrs = [0.0, 6.0, 12.0, 16.0]
    rf, target, budget = 2048, 100, 4 * 2048 * 192
    kw = dict(noise="complex", snr_def="esn0")
    got, rounds = ofdm.mc_sweep_channel_until(SEED, 0, 2, snrs, pkg.MODE_EXACT, target_errors=target, max_bits=budget, round_frames=rf, **kw)
    assert rounds == 4 and got[0].frames == rf and got[-1].frames == 4 * rf    # 0 dB is done after one round, 16 dB runs to the budget
    for c in got:
        assert c.bit_errors >= target or c.bits >= budget
    a, r1 = pkg.sweep.mc_sweep_until(ofdm, SEED, 2, snrs, pkg.MODE_EXACT, target, budget, rf, **kw)
    assert r1 == rounds and [ints(x) for x in a] == [ints(x) for x in got]

    def two_ranks(points, lo, n):
        tot_i = np.zeros((len(points), 5), np.int64); tot_d = np.zeros((len(points), 3), np.float64)
        for rank in range(2):
            l2, h2 = pkg.sweep.shard_range(n, rank, 2)
            c = ofdm.new_counters(len(points))
            ofdm.mc_sweep_channel(SEED, lo + l2, h2 - l2, 2, [snrs[p] for p in points], pkg.MODE_EXACT, streams=points, counters=c, **kw)
            raw = c.cpu().numpy()
            tot_i += raw[:, :5]; tot_d += raw[:, 5:].copy().view(np.float64)
        return tot_i, tot_d
    i2, _, r2 = pkg.sweep.until_loop(two_ranks, len(snrs), target, budget, rf)
    assert r2 == rounds and [tuple(int(v) for v in row) for row in i2] == [ints(x) for x in got]


# ---- 6. statistics of the complex / Es/N0 curve
def test_complex_esn0_statistics(ofdm, pkg):
    n_gpu, n_model, chunk = 1 << 22, 1 << 20, 1 << 16
    snrs = [0.0, 2.0, 4.0, 6.0, 8.0, 10.0]
    got = ofdm.mc_sweep_channel(SEED, 0, n_gpu, 2, snrs, pkg.MODE_FAST, "complex", "esn0")
    textbook = pkg.sweep.qpsk_ber_awgn(snrs, "esn0")
    rng = np.random.default_rng(2024)
    for i, s in enumerate(snrs):
        fe = np.concatenate([model_complex_esn0(s, chunk, 2, rng) for _ in range(n_model // chunk)]).astype(np.float64)
        for stat, gpu_mean in ((fe / 192.0, got[i].bit_errors / got[i].bits), ((fe > 0).astype(np.float64), got[i].frames_in_error / got[i].frames)):
            m, v = stat.mean(), stat.var(ddof=1)
            se = math.sqrt(v / n_model + v / n_gpu)            # per-frame variance of the model, for both sample sizes
            assert abs(gpu_mean - m) <= 4.0 * se, (s, gpu_mean, m, se)
        assert got[i].bit_errors / got[i].bits > textbook[i], (s, got[i].bit_errors / got[i].bits, textbook[i])


# ---- 7. the C driver
def test_c_driver_channel(ofdm, pkg, tmp_path):
    from conftest import ROOT
    exe = os.path.join(ROOT, "ieee-802.11-ofdm-qpsk-simulator_b200", "ofdm_sweep")
    if not os.path.exists(exe):
        import __graft_entry__ as entry
        entry.build()
    out = tmp_path / "data"; out.mkdir()
    r = subprocess.run([exe, "--quiet", "--outdir", str(out), "--frames", "65536", "--noise", "complex", "--snr-def", "esn0", "--mode", "exact",
                        "--snr-start", "0", "--snr-step", "2", "--snr-count", "5", "--seed", "3"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    snrs = [0.0, 2.0, 4.0, 6.0, 8.0]
    want = ofdm.mc_sweep_channel(3, 0, 65536, 2, snrs, pkg.MODE_EXACT, "complex", "esn0")
    text = "\t".join("%.2e" % np.float32(ofdm.finalize(c)[2]) for c in want) + "\n"
    assert open(out / "Output_BER.txt").read() == text
    r = subprocess.run([exe, "--quiet", "--outdir", str(out), "--noise", "complex", "--draws", os.devnull], capture_output=True, text=True, timeout=60)
    assert r.returncode != 0 and "--draws" in r.stderr


# ---- 8. invalid channels
def test_invalid_channels(ofdm, pkg, lib):
    snr = np.zeros(2, np.float32)
    cnt = ofdm.new_counters(2)
    out = (pkg.Counters * 2)()
    rounds = C.c_int(0)
    h = ofdm.h
    for ch in (None, pkg.Channel(2, 0, 0), pkg.Channel(-1, 0, 0), pkg.Channel(1, 3, 0), pkg.Channel(0, -1, 0), pkg.Channel(1, 1, 17),
               pkg.Channel(1, 1, -1)):
        ref = None if ch is None else C.byref(ch)
        assert lib.ofdm_mc_sweep_channel_dev(h, ref, SEED, 0, 64, 2, snr.ctypes.data, None, 2, 0, cnt.data_ptr()) == 1
        assert lib.ofdm_mc_sweep_channel_until(h, ref, SEED, 0, 2, snr.ctypes.data, 2, 0, 100, 1000, 64, out, C.byref(rounds)) == 1
    tx = ofdm.zeros((4, 320, 2), ofdm.torch.float32)
    ota = ofdm.zeros((4, 320, 2), ofdm.torch.float32)
    for noise, snr_def in ((2, 0), (0, 3), (-1, 1)):
        assert lib.ofdm_awgn_philox_ex(h, noise, snr_def, tx.data_ptr(), None, 3.0, SEED, 0, 0, ota.data_ptr(), 4, 2, 0) == 1
    # the context is still usable
    got = ofdm.mc_sweep_channel(SEED, 0, 256, 2, [3.0], pkg.MODE_EXACT, "complex", "esn0")
    assert got[0].frames == 256
