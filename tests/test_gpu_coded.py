"""The coded link on the GPU (include/ofdm_b200.h "the coded link", DESIGN.md section 6.2): k_conv_encode and k_viterbi bit for bit
against the CPU oracle on the GPU's own inputs, the EXACT coded sweeps against the oracle's whole coded chain on the GPU's draws,
the FAST route against EXACT, split invariance and the until rule over ranks, the statistics of an independent float64 model,
the kernels a coded sweep launches, argument errors and the C driver's --code."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from coded_oracle import CodedOracle, k_info, np_inputs, np_viterbi

pytestmark = pytest.mark.gpu

SEED = 41
RATES = ["1/2", "3/4"]
DECISIONS = ["soft", "hard"]
SNR_UNIT_COMPLEX = -21.072099685668945        # the Es/N0 point whose noise power is exactly 2.0f: sigma = 1 per rail


def ints(c):
    return (int(c.bit_errors), int(c.bits), int(c.frames_in_error), int(c.rail_errors), int(c.frames))


@pytest.fixture(scope="module")
def co():
    return CodedOracle()


def info_bits(ofdm, pkg, words, n_sym):
    return pkg.unpack_bits_host(words.cpu().numpy().view(np.uint32).reshape(-1, 3 * n_sym))


def gpu_draws(ofdm, pkg, stream, frame0, n_frames, n_sym):
    """the GPU's domain-0 and domain-4 normals of (SEED, stream), bit for bit (the channel on all-zero frames, sigma = 1)"""
    zeros = ofdm.zeros((n_frames, pkg.frame_len(n_sym), 2), ofdm.torch.float32)
    c = ofdm.awgn_philox_ex(zeros, SNR_UNIT_COMPLEX, SEED, stream, frame0, n_sym, pkg.MODE_EXACT, "complex", "esn0").cpu().numpy()
    return c[..., 0].copy(), c[..., 1].copy()


def received(ofdm, pkg, payload, n_sym, snr, stream, frame0, n_taps=0, mode=None):
    """transmitter -> [taps] -> complex Es/N0 channel -> receiver with H and eq dumps"""
    mode = pkg.MODE_EXACT if mode is None else mode
    tx = ofdm.tx_frames(payload, n_sym, mode, with_power=False)
    if n_taps:
        tx, _ = ofdm.multipath_philox(tx, SEED, frame0, n_taps, n_sym)
    ota = ofdm.awgn_philox_ex(tx, snr, SEED, stream, frame0, n_sym, mode, "complex", "esn0")
    raw, bufs = ofdm.rx_frames(ota, payload, n_sym, mode, want=("H", "eq"))
    return raw, bufs["H"], bufs["eq"]


# ---- 1. the encoder
@pytest.mark.parametrize("rate", RATES)
@pytest.mark.parametrize("n_sym", [1, 2, 5, 512])
def test_encode_matches_oracle(ofdm, pkg, co, rate, n_sym):
    n = 5 if n_sym == 512 else 301
    words = ofdm.random_bits(SEED, 77, n, n_sym)
    got = ofdm.conv_encode(words, n_sym, rate).cpu().numpy().view(np.uint32).reshape(n, -1)
    want = pkg.pack_bits_host(co.conv_encode(info_bits(ofdm, pkg, words, n_sym), n_sym, rate))
    assert np.array_equal(got, want)


# ---- 2. the decoder on the GPU's own dumps
def check_decode(ofdm, pkg, co, words, H, eq, n_sym, rate, decision):
    cnt, dec = ofdm.viterbi_decode(H, eq, n_sym, rate, decision, info=words)
    n = H.shape[0]
    want_bits = co.viterbi(H.cpu().numpy(), eq.cpu().numpy(), n_sym, rate, decision)
    full = np.zeros((n, 96 * n_sym), np.uint8)
    full[:, :want_bits.shape[1]] = want_bits
    assert np.array_equal(dec.cpu().numpy().view(np.uint32).reshape(n, -1), pkg.pack_bits_host(full)), (rate, decision, n_sym)
    info = info_bits(ofdm, pkg, words, n_sym)[:, :k_info(rate, n_sym)]
    fe = (want_bits != info).sum(axis=1)
    assert ints(cnt) == (int(fe.sum()), n * k_info(rate, n_sym), int((fe > 0).sum()), 0, n)
    assert cnt.sum_err2 == 0 and cnt.sum_ref2 == 0 and cnt.sum_evm_lin == 0
    return fe


@pytest.mark.parametrize("decision", DECISIONS)
@pytest.mark.parametrize("rate", RATES)
@pytest.mark.parametrize("n_sym", [1, 2, 3, 37, 512])
def test_decode_matches_oracle(ofdm, pkg, co, n_sym, rate, decision):
    n = 3 if n_sym == 512 else 24 if n_sym == 37 else 200
    words = ofdm.random_bits(SEED, 500, n, n_sym)
    payload = ofdm.conv_encode(words, n_sym, rate)
    total = 0
    for stream, snr in enumerate((-1.0, 3.0, 7.0)):
        _, H, eq = received(ofdm, pkg, payload, n_sym, snr, stream, 500)
        total += check_decode(ofdm, pkg, co, words, H, eq, n_sym, rate, decision).sum()
    assert total > 0                                            # the low point has errors left to decode


@pytest.mark.parametrize("decision", DECISIONS)
@pytest.mark.parametrize("rate", RATES)
def test_decode_with_taps_and_erasures(ofdm, pkg, co, rate, decision):
    n, n_sym = 160, 3
    words = ofdm.random_bits(SEED, 900, n, n_sym)
    payload = ofdm.conv_encode(words, n_sym, rate)
    for stream, snr in enumerate((4.0, 10.0)):
        _, H, eq = received(ofdm, pkg, payload, n_sym, snr, stream, 900, n_taps=4)
        check_decode(ofdm, pkg, co, words, H, eq, n_sym, rate, decision)
        # a faded-out data bin: H = 0 there, and the equaliser's F / 0 in eq (inf or NaN) -- an erasure of the soft decoder
        H2, eq2 = H.clone(), eq.clone()
        H2[::2, 20] = 0.0                                       # centred bin 20 = data point 13
        eq2[::2, 13::48, 0] = float("inf")
        eq2[::2, 13::48, 1] = float("nan")
        check_decode(ofdm, pkg, co, words, H2, eq2, n_sym, rate, decision)


@pytest.mark.parametrize("rate,max_flips", [("1/2", 4), ("3/4", 2)])
def test_synthetic_flips_decode_clean(ofdm, pkg, co, rate, max_flips):
    n, n_sym = 400, 2
    words = ofdm.random_bits(SEED, 3, n, n_sym)
    payload = pkg.unpack_bits_host(ofdm.conv_encode(words, n_sym, rate).cpu().numpy().view(np.uint32).reshape(n, -1)).astype(np.int64)
    p = payload.reshape(n, n_sym * 48, 2)
    c1 = 1 - p[..., 0]
    c0 = p[..., 1] ^ c1
    eq = np.stack([2 * c0 - 1, 2 * c1 - 1], axis=-1).astype(np.float32)
    rng = np.random.default_rng(9)
    for f in range(n):
        k = int(rng.integers(0, max_flips + 1))
        eq[f].reshape(-1)[rng.choice(96 * n_sym, size=k, replace=False)] *= -1
    H = np.zeros((n, 64, 2), np.float32)
    H[..., 0] = 1.0
    for decision in DECISIONS:
        cnt, _ = ofdm.viterbi_decode(ofdm.to_dev(H), ofdm.to_dev(eq), n_sym, rate, decision, info=words)
        assert cnt.bit_errors == 0 and cnt.frames == n


# ---- 3. EXACT coded sweeps against the oracle's whole coded chain
CHANNELS = [("real", "frame_power"), ("complex", "esn0"), ("complex", "ebn0")]


def oracle_coded_sweep(ofdm, pkg, co, frame0, n, n_sym, snrs, noise, snr_def, n_taps, rate, decision):
    info = co.philox_bits(SEED, frame0, n, n_sym)
    taps = None
    if n_taps:
        tx = ofdm.tx_frames(ofdm.random_bits(SEED, frame0, n, n_sym), n_sym, pkg.MODE_EXACT, with_power=False)
        taps = ofdm.multipath_philox(tx, SEED, frame0, n_taps, n_sym)[1].cpu().numpy()        # the GPU's own taps
    out = []
    for i, s in enumerate(snrs):
        g0, g1 = gpu_draws(ofdm, pkg, i, frame0, n, n_sym)
        out.append(co.coded_chain(info, g0, g1 if noise == "complex" else None, taps, n_sym, s, noise, snr_def, rate, decision))
    return out


@pytest.mark.parametrize("n_taps", [0, 4])
@pytest.mark.parametrize("noise,snr_def", CHANNELS)
@pytest.mark.parametrize("decision", DECISIONS)
@pytest.mark.parametrize("rate", RATES)
def test_exact_coded_sweep_against_oracle(ofdm, pkg, co, rate, decision, noise, snr_def, n_taps):
    n, frame0, n_sym = 211, 333, 2
    snrs = [0.0, 3.0] if snr_def != "frame_power" else [2.0, 6.0]
    want = oracle_coded_sweep(ofdm, pkg, co, frame0, n, n_sym, snrs, noise, snr_def, n_taps, rate, decision)
    coded, raw = ofdm.mc_sweep_coded(SEED, frame0, n, n_sym, snrs, pkg.MODE_EXACT, rate, decision, noise, snr_def, n_taps)
    for g, r, (wc, wr) in zip(coded, raw, want):
        assert ints(g) == ints(wc), (ints(g), ints(wc))
        assert ints(r) == ints(wr), (ints(r), ints(wr))
        assert abs(r.sum_err2 - wr.sum_err2) <= 1e-5 * wr.sum_err2 and abs(r.sum_evm_lin - wr.sum_evm_lin) <= 1e-5 * wr.sum_evm_lin
    assert sum(c.bit_errors for c in coded) > 0


@pytest.mark.parametrize("rate", RATES)
def test_fast_agrees_with_exact(ofdm, pkg, rate):
    n, snrs = 20000, [1.0, 3.0, 5.0]
    for noise, snr_def in (("complex", "ebn0"), ("real", "frame_power")):
        fc, fr = ofdm.mc_sweep_coded(SEED, 0, n, 2, snrs, pkg.MODE_FAST, rate, "soft", noise, snr_def)
        ec, er = ofdm.mc_sweep_coded(SEED, 0, n, 2, snrs, pkg.MODE_EXACT, rate, "soft", noise, snr_def)
        for a, b in zip(fc, ec):
            assert (a.bits, a.frames) == (b.bits, b.frames)
            # fp32 transforms move a few decoder inputs by an ulp-scale amount: a handful of packets may decode differently
            assert abs(int(a.frames_in_error) - int(b.frames_in_error)) <= 3 + 1e-3 * b.frames_in_error
            assert abs(int(a.bit_errors) - int(b.bit_errors)) <= 30 + 1e-3 * b.bit_errors
        for a, b in zip(fr, er):
            assert abs(int(a.rail_errors) - int(b.rail_errors)) <= 2 + 1e-5 * b.rail_errors


def test_raw_rail_errors_are_the_coded_bit_errors(ofdm, pkg):
    n, n_sym, snrs = 3000, 2, [0.0, 4.0]
    for rate in RATES:
        coded, raw = ofdm.mc_sweep_coded(SEED, 10, n, n_sym, snrs, pkg.MODE_EXACT, rate, "hard", "complex", "esn0")
        words = ofdm.random_bits(SEED, 10, n, n_sym)
        payload = ofdm.conv_encode(words, n_sym, rate)
        p = pkg.unpack_bits_host(payload.cpu().numpy().view(np.uint32).reshape(n, -1)).astype(np.int64).reshape(n, n_sym * 48, 2)
        c1 = 1 - p[..., 0]
        c0 = p[..., 1] ^ c1
        for i, s in enumerate(snrs):
            _, _, eq = received(ofdm, pkg, payload, n_sym, s, i, 10)
            e = eq.cpu().numpy()
            wrong = int(((e[..., 0] > 0) != (c0 == 1)).sum() + ((e[..., 1] > 0) != (c1 == 1)).sum())
            assert raw[i].rail_errors == wrong and wrong > 0


# ---- 4. split invariance and the until rule over ranks
def test_split_chunk_invariance(ofdm, pkg):
    snrs = [1.0, 3.0, 5.0]
    for rate, n_sym in (("1/2", 2), ("3/4", 3)):
        kw = dict(rate=rate, decision="soft", noise="complex", snr_def="ebn0")
        whole, wraw = ofdm.mc_sweep_coded(SEED, 1000, 2000, n_sym, snrs, pkg.MODE_EXACT, **kw)
        parts = [ofdm.mc_sweep_coded(SEED, 1000 + off, k, n_sym, snrs, pkg.MODE_EXACT, **kw) for off, k in ((0, 700), (700, 1), (701, 1299))]
        for i in range(len(snrs)):
            assert tuple(sum(ints(p[0][i])[k] for p in parts) for k in range(5)) == ints(whole[i])
            assert tuple(sum(ints(p[1][i])[k] for p in parts) for k in range(5)) == ints(wraw[i])
        last, _ = ofdm.mc_sweep_coded(SEED, 1000, 2000, n_sym, snrs[2:], pkg.MODE_EXACT, streams=[2], **kw)
        assert ints(last[0]) == ints(whole[2])
    # 512-symbol frames run in chunks of the staged route and keep their survivors in HBM
    a, _ = ofdm.mc_sweep_coded(SEED, 7, 6, 512, [2.0], pkg.MODE_EXACT, "3/4", "soft", "complex", "ebn0")
    b = [ofdm.mc_sweep_coded(SEED, 7 + k, 1, 512, [2.0], pkg.MODE_EXACT, "3/4", "soft", "complex", "ebn0")[0][0] for k in range(6)]
    assert tuple(sum(ints(x)[k] for x in b) for k in range(5)) == ints(a[0])


def test_until_rule_over_ranks(ofdm, pkg):
    snrs = [0.0, 2.0, 4.0, 6.0]
    rf, target, budget = 2048, 100, 4 * 2048 * 90
    kw = dict(rate="1/2", decision="soft", noise="complex", snr_def="ebn0")
    coded, raw, rounds = ofdm.mc_sweep_coded_until(SEED, 0, 2, snrs, pkg.MODE_EXACT, target_errors=target, max_bits=budget, round_frames=rf, **kw)
    for c in coded:
        assert c.bit_errors >= target or c.bits >= budget
    assert coded[0].frames == rf and coded[-1].frames > rf and [c.frames for c in raw] == [c.frames for c in coded]
    a, r1 = pkg.sweep.mc_sweep_until(ofdm, SEED, 2, snrs, pkg.MODE_EXACT, target, budget, rf, noise="complex", snr_def="ebn0", code="1/2")
    assert r1 == rounds and [ints(x) for x in a] == [ints(x) for x in coded]

    def two_ranks(points, lo, n):
        tot_i = np.zeros((len(points), 5), np.int64); tot_d = np.zeros((len(points), 3), np.float64)
        for rank in range(2):
            l2, h2 = pkg.sweep.shard_range(n, rank, 2)
            c = ofdm.new_counters(len(points))
            ofdm.mc_sweep_coded(SEED, lo + l2, h2 - l2, 2, [snrs[p] for p in points], pkg.MODE_EXACT, streams=points, counters=(c, None), **kw)
            raw_ = c.cpu().numpy()
            tot_i += raw_[:, :5]; tot_d += raw_[:, 5:].copy().view(np.float64)
        return tot_i, tot_d
    i2, _, r2 = pkg.sweep.until_loop(two_ranks, len(snrs), target, budget, rf)
    assert r2 == rounds and [tuple(int(v) for v in row) for row in i2] == [ints(x) for x in coded]


# ---- 5. statistics against an independent float64 model
def model_coded_ebn0(ebn0_db, rate, n_frames, n_sym, rng):
    """per-frame information-bit errors of the complex / Eb/N0 coded link, written from the definitions alone: np = 1 / (64 2R Eb/N0),
    a data bin carries X + CN(0, 64 np), the LTS estimate H = 1 + CN(0, 32 np) per data bin (the same for the frame), the soft
    decoder input conj(H) F per rail; the code, the interleaver and a float64 Viterbi as in coded_oracle.np_*"""
    from coded_oracle import np_encode
    R = 0.5 if rate == "1/2" else 0.75
    npow = 1.0 / (64.0 * 2.0 * R * 10.0 ** (ebn0_db / 10.0))
    K = k_info(rate, n_sym)
    info = rng.integers(0, 2, (n_frames, K))
    coded = np_encode(info, rate, n_sym).astype(np.int64).reshape(n_frames, n_sym, 96)
    k = np.arange(96)
    pos = np.zeros_like(coded)
    pos[:, :, 6 * (k % 16) + k // 16] = coded                  # interleaver: position of coded bit k
    pos = pos.reshape(n_frames, n_sym, 48, 2)
    X = ((2 * pos[..., 0] - 1) + 1j * (2 * pos[..., 1] - 1)) / np.sqrt(2.0)

    def cn(var, shape):
        return np.sqrt(var / 2.0) * (rng.standard_normal(shape) + 1j * rng.standard_normal(shape))
    Hd = 1.0 + cn(32.0 * npow, (n_frames, 1, 48))
    F = X + cn(64.0 * npow, X.shape)
    Y = np.conj(Hd) * F
    H = np.zeros((n_frames, 64, 2))
    H[..., 0] = 1.0                                              # w = 1: Y already carries |H|^2 eq = conj(H) F
    eq = np.stack([Y.real, Y.imag], axis=-1).reshape(n_frames, n_sym * 48, 2)
    La, Lb = np_inputs(H, eq, n_sym, rate, "soft")
    bits, _ = np_viterbi(La, Lb)
    return (bits[:, :K] != info).sum(axis=1)


def test_coded_statistics_against_model(ofdm, pkg):
    n_gpu, n_model, chunk, n_sym = 1 << 21, 24000, 4000, 2
    snrs = [1.0, 2.0, 3.0]
    for rate in RATES:
        got, _ = ofdm.mc_sweep_coded(SEED, 0, n_gpu, n_sym, snrs, pkg.MODE_FAST, rate, "soft", "complex", "ebn0")
        rng = np.random.default_rng(77)
        K = k_info(rate, n_sym)
        for i, s in enumerate(snrs):
            fe = np.concatenate([model_coded_ebn0(s, rate, chunk, n_sym, rng) for _ in range(n_model // chunk)]).astype(np.float64)
            # errors come in bursts within a packet: the spread is the per-frame variance, not a binomial one
            for stat, gpu_mean in ((fe / K, got[i].bit_errors / got[i].bits), ((fe > 0).astype(np.float64), got[i].frames_in_error / got[i].frames)):
                m, v = stat.mean(), stat.var(ddof=1)
                se = math.sqrt(v / n_model + v / n_gpu)
                assert abs(gpu_mean - m) <= 4.0 * se, (rate, s, gpu_mean, m, se)


def test_soft_beats_hard_and_coded_beats_uncoded(ofdm, pkg):
    n, s = 1 << 20, [4.0]
    uncoded = ofdm.mc_sweep_channel(SEED, 0, n, 2, s, pkg.MODE_FAST, "complex", "ebn0")[0]
    for rate in RATES:
        soft = ofdm.mc_sweep_coded(SEED, 0, n, 2, s, pkg.MODE_FAST, rate, "soft", "complex", "ebn0")[0][0]
        hard = ofdm.mc_sweep_coded(SEED, 0, n, 2, s, pkg.MODE_FAST, rate, "hard", "complex", "ebn0")[0][0]
        ber = lambda c: c.bit_errors / c.bits                      # noqa: E731
        assert ber(soft) < 0.5 * ber(hard), (rate, ber(soft), ber(hard))
        assert ber(soft) < 0.5 * ber(uncoded), (rate, ber(soft), ber(uncoded))
        assert soft.frames_in_error < hard.frames_in_error


# ---- 6. what one coded sweep launches
KERNELS_SCRIPT = """
import json, sys
import __graft_entry__ as entry
from test_gpu_routes import observe
pkg = entry.load_pkg()
o = pkg.Ofdm(0)
snrs = [1.0, 2.0, 3.0]
cnt = (o.new_counters(3), o.new_counters(3))
call = lambda: o.mc_sweep_coded(41, 0, 4096, 2, snrs, pkg.MODE_FAST, "1/2", "soft", "complex", "esn0", counters=cnt)
call()
kernels, launches, _ = observe(o, call)
print(json.dumps({"kernels": kernels, "launches": launches}))
"""


def test_coded_sweep_kernels():
    """the route tests' profiler harness (torch.profiler kernel names in launch order, ofdm_ctx_launch_count), in a process of its
    own so that this profiler session cannot leave activity records behind for the route tests' sessions"""
    import json
    import sys
    from conftest import ROOT
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, here, os.environ.get("PYTHONPATH", "")]))
    r = subprocess.run([sys.executable, "-c", KERNELS_SCRIPT], cwd=here, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    got = json.loads(r.stdout.strip().splitlines()[-1])
    kernels = got["kernels"]
    # bits, encoder, transmitter; per point the channel, the dumping receiver and the decoder
    assert got["launches"] == len(kernels) == 3 + 3 * 3
    assert [k.split("<")[0] for k in kernels] == ["k_philox_bits", "k_conv_encode", "k_tx_frames2"] + ["k_awgn_channel", "k_rx_frames", "k_viterbi"] * 3, kernels


# ---- 7. argument errors
def test_argument_errors(ofdm, pkg, lib):
    h = ofdm.h
    snr = np.zeros(2, np.float32)
    c2 = ofdm.new_counters(2)
    out = (pkg.Counters * 2)()
    rounds = C.c_int(0)
    words = ofdm.random_bits(SEED, 0, 4, 2)
    pay = ofdm.empty((24,), ofdm.torch.int32)
    H = ofdm.zeros((4, 64, 2), ofdm.torch.float32)
    eq = ofdm.zeros((4, 96, 2), ofdm.torch.float32)
    ch = pkg.channel("complex", "esn0")
    for rate in (0, 3, -1):
        assert lib.ofdm_conv_encode(h, rate, words.data_ptr(), pay.data_ptr(), 4, 2) == 1
    assert lib.ofdm_conv_encode(h, 1, words.data_ptr(), pay.data_ptr(), 4, 0) == 1
    assert lib.ofdm_conv_encode(h, 1, words.data_ptr(), pay.data_ptr(), 4, 513) == 1
    assert lib.ofdm_conv_encode(h, 1, None, pay.data_ptr(), 4, 2) == 1
    assert lib.ofdm_conv_encode(h, 1, words.data_ptr(), pay.data_ptr(), -1, 2) == 1
    bad_codes = [None, pkg.Code(0, 0), pkg.Code(3, 0), pkg.Code(1, 2), pkg.Code(2, -1)]
    for cd in bad_codes:
        ref = None if cd is None else C.byref(cd)
        assert lib.ofdm_viterbi_decode(h, ref, H.data_ptr(), eq.data_ptr(), None, None, 4, 2, None) == 1
        assert lib.ofdm_mc_sweep_coded_dev(h, C.byref(ch), ref, SEED, 0, 64, 2, snr.ctypes.data, None, 2, 0, c2.data_ptr(), None) == 1
        assert lib.ofdm_mc_sweep_coded_until(h, C.byref(ch), ref, SEED, 0, 2, snr.ctypes.data, 2, 0, 100, 1000, 64, out, None, C.byref(rounds)) == 1
    good = pkg.code("1/2", "soft")
    assert lib.ofdm_viterbi_decode(h, C.byref(good), None, eq.data_ptr(), None, None, 4, 2, None) == 1
    assert lib.ofdm_viterbi_decode(h, C.byref(good), H.data_ptr(), eq.data_ptr(), None, None, 4, 2, c2.data_ptr()) == 1   # counting needs info
    assert lib.ofdm_viterbi_decode(h, C.byref(good), H.data_ptr(), eq.data_ptr(), None, None, 4, 0, None) == 1
    for bad_ch in (None, pkg.Channel(2, 0, 0), pkg.Channel(1, 3, 0), pkg.Channel(1, 1, 17)):
        ref = None if bad_ch is None else C.byref(bad_ch)
        assert lib.ofdm_mc_sweep_coded_dev(h, ref, C.byref(good), SEED, 0, 64, 2, snr.ctypes.data, None, 2, 0, c2.data_ptr(), None) == 1
        assert lib.ofdm_mc_sweep_coded_until(h, ref, C.byref(good), SEED, 0, 2, snr.ctypes.data, 2, 0, 100, 1000, 64, out, None, C.byref(rounds)) == 1
    assert lib.ofdm_mc_sweep_coded_dev(h, C.byref(ch), C.byref(good), SEED, 0, 64, 2, snr.ctypes.data, None, 2, 2, c2.data_ptr(), None) == 1   # mode
    assert lib.ofdm_mc_sweep_coded_dev(h, C.byref(ch), C.byref(good), SEED, 0, 64, 2, snr.ctypes.data, None, 2, 0, None, None) == 1
    assert lib.ofdm_mc_sweep_coded_dev(h, C.byref(ch), C.byref(good), SEED, 0, 64, 2, snr.ctypes.data, None, 65, 0, c2.data_ptr(), None) == 1
    assert lib.ofdm_mc_sweep_coded_until(h, C.byref(ch), C.byref(good), SEED, 0, 2, snr.ctypes.data, 2, 0, 100, 1000, 0, out, None, C.byref(rounds)) == 1
    with pytest.raises(ValueError):
        pkg.code("2/3")
    with pytest.raises(ValueError):
        pkg.code("1/2", "erasure")
    got, _ = ofdm.mc_sweep_coded(SEED, 0, 256, 2, [3.0], pkg.MODE_EXACT, "1/2", "soft", "complex", "esn0")       # still usable
    assert got[0].frames == 256


# ---- 8. the C driver
def run_driver(args, timeout=900):
    from conftest import ROOT
    exe = os.path.join(ROOT, "ieee-802.11-ofdm-qpsk-simulator_b200", "ofdm_sweep")
    if not os.path.exists(exe):
        import __graft_entry__ as entry
        entry.build()
    return subprocess.run([exe, "--quiet"] + args, capture_output=True, text=True, timeout=timeout)


def test_c_driver_code(ofdm, pkg, tmp_path):
    import torch
    snrs = [0.0, 1.0, 2.0, 3.0]
    common = ["--noise", "complex", "--snr-def", "ebn0", "--mode", "exact", "--snr-start", "0", "--snr-step", "1", "--snr-count", "4", "--seed", "3"]
    outs = {}
    for gpus in (1, 2) if torch.cuda.device_count() >= 2 else (1,):
        out = tmp_path / ("g%d" % gpus); out.mkdir()
        r = run_driver(["--outdir", str(out), "--frames", "40000", "--code", "3/4", "--decision", "soft", "--gpus", str(gpus)] + common)
        assert r.returncode == 0, r.stdout + r.stderr
        assert "code 3/4 soft" in r.stderr
        outs[gpus] = {f: open(out / f, "rb").read() for f in ("Output_SNR.txt", "Output_BER.txt", "Output_PER.txt", "Output_EVM_AGC.txt", "Output_EVM_AGC_DB.txt")}
    coded, raw = ofdm.mc_sweep_coded(3, 0, 40000, 2, snrs, pkg.MODE_EXACT, "3/4", "soft", "complex", "ebn0")
    assert outs[1]["Output_BER.txt"].decode() == "\t".join("%.2e" % np.float32(c.bit_errors / c.bits) for c in coded) + "\n"
    assert outs[1]["Output_PER.txt"].decode() == "\t".join("%.2e" % np.float32(c.frames_in_error / c.frames) for c in coded) + "\n"
    assert outs[1]["Output_EVM_AGC.txt"].decode() == "\t".join("%.2e" % np.float32(ofdm.finalize(c)[0]) for c in raw) + "\n"
    if 2 in outs:
        assert outs[2] == outs[1]
    # the until rule on the coded counters
    out = tmp_path / "until"; out.mkdir()
    r = run_driver(["--outdir", str(out), "--target-errors", "200", "--round-frames", "8192", "--code", "1/2"] + common)
    assert r.returncode == 0, r.stdout + r.stderr
    want, _, _ = ofdm.mc_sweep_coded_until(3, 0, 2, snrs, pkg.MODE_EXACT, "1/2", "soft", "complex", "ebn0", target_errors=200,
                                          max_bits=200 * 10 ** 7, round_frames=8192)
    assert open(out / "Output_PER.txt").read() == "\t".join("%.2e" % np.float32(c.frames_in_error / c.frames) for c in want) + "\n"
    for bad in (["--message", "hi", "--code", "1/2"], ["--draws", os.devnull, "--code", "1/2"], ["--frames", "100", "--code", "2/3"],
                ["--frames", "100", "--decision", "hard"]):
        r = run_driver(["--outdir", str(out)] + bad, timeout=60)
        assert r.returncode != 0, bad
