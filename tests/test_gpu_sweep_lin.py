"""k_sweep_lin: the whole injected-noise SNR sweep in one kernel (FFT(x + sigma g) = FFT(x) + sigma FFT(g), csrc/ofdm_sweep.cuh).
The totals must be those of the one-launch-per-SNR-point route and, in EXACT mode, those of the reference: checked against
the CPU oracle, the all-exact kernels and a run in which every (frame, SNR point) is replayed, on ordinary, ragged and
adversarial inputs."""
import numpy as np
import pytest

from conftest import bits_and_noise

pytestmark = pytest.mark.gpu

SNR21 = [float(s) for s in range(21)]


def ints(c):
    return (c.bit_errors, c.bits, c.frames_in_error, c.rail_errors, c.frames)


@pytest.fixture()
def knobs(ofdm):
    yield ofdm
    for name, v in (("fused_sweep", 1), ("exact_speculation", 1), ("force_replay", 0), ("force_generic_rx", 0)):
        ofdm.set_option(name, v)


@pytest.mark.parametrize("n_frames", [1, 2, 3, 31, 777, 5000])
def test_fused_equals_per_point_and_oracle(knobs, pkg, port, n_frames):
    ofdm = knobs
    bits, g = bits_and_noise(1300 + n_frames, n_frames, 2)
    packed = ofdm.to_dev(pkg.pack_bits_host(bits).view(np.int32))
    gd = ofdm.to_dev(g)
    snr = [0.0, 3.0, 7.5, 12.0, 30.0]
    fused = ofdm.sweep_inject_dev(packed, gd, n_frames, 2, snr, pkg.MODE_EXACT)
    ofdm.set_option("fused_sweep", 0)
    staged = ofdm.sweep_inject_dev(packed, gd, n_frames, 2, snr, pkg.MODE_EXACT)
    ofdm.set_option("fused_sweep", 1)
    want = port.chain_sweep(bits, g, 2, snr)
    for a, b, w in zip(fused, staged, want):
        assert ints(a) == ints(b) == (w.bit_errors, w.bits, w.frames_in_error, w.rail_errors, w.frames)
        assert abs(a.sum_err2 / a.sum_ref2 - w.sum_err2 / w.sum_ref2) <= 1e-5 * w.sum_err2 / w.sum_ref2
        assert abs(a.sum_evm_lin - w.sum_evm_lin) <= 1e-5 * w.sum_evm_lin
    # fast mode: the same decisions up to rails within fp32 rounding of zero, EVM within 1e-5 (small-|H| bins are replayed)
    fast = ofdm.sweep_inject_dev(packed, gd, n_frames, 2, snr, pkg.MODE_FAST)
    for a, w in zip(fast, want):
        assert abs(int(a.bit_errors) - int(w.bit_errors)) <= 2 and a.frames == w.frames
        assert abs(a.sum_err2 / a.sum_ref2 - w.sum_err2 / w.sum_ref2) <= 1e-5 * w.sum_err2 / w.sum_ref2


@pytest.mark.parametrize("n_snr", [21, 33, 64, 70])
def test_many_snr_points(knobs, pkg, port, n_snr):
    """SNR points beyond 32 live in the lanes' second slot, beyond 64 in a second launch"""
    ofdm = knobs
    n_frames = 600
    bits, g = bits_and_noise(77 + n_snr, n_frames, 2)
    packed = ofdm.to_dev(pkg.pack_bits_host(bits).view(np.int32))
    gd = ofdm.to_dev(g)
    snr = list(np.linspace(-3.0, 24.0, n_snr).astype(np.float32))
    fused = ofdm.sweep_inject_dev(packed, gd, n_frames, 2, snr, pkg.MODE_EXACT)
    want = port.chain_sweep(bits, g, 2, snr)
    for a, w in zip(fused, want):
        assert ints(a) == (w.bit_errors, w.bits, w.frames_in_error, w.rail_errors, w.frames)


def test_every_point_replayed_and_all_exact(knobs, pkg):
    ofdm = knobs
    import torch
    n = 120_000
    gen = torch.Generator(device=ofdm.device); gen.manual_seed(41)
    packed = torch.randint(-2 ** 31, 2 ** 31 - 1, (n * 6,), dtype=torch.int32, device=ofdm.device, generator=gen)
    g = torch.randn((n, 320), dtype=torch.float32, device=ofdm.device, generator=gen)
    snr = [-6.0, 0.0, 2.0, 6.0, 10.0, 14.0]
    runs = {}
    for name, fused, spec, force in (("fused", 1, 1, 0), ("replay_all", 1, 1, 1), ("all_exact", 0, 0, 0), ("staged_checked", 0, 1, 0)):
        ofdm.set_option("fused_sweep", fused); ofdm.set_option("exact_speculation", spec); ofdm.set_option("force_replay", force)
        ofdm.replayed_frames(reset=True)
        runs[name] = (ofdm.sweep_inject_dev(packed, g, n, 2, snr, pkg.MODE_EXACT), ofdm.replayed_frames())
    # the fp32 sweep kernel's EVM-guard replay, forced for every point, on the same (exact) transmitter frames
    ofdm.set_option("fused_sweep", 1); ofdm.set_option("exact_speculation", 1); ofdm.set_option("force_replay", 1)
    frames, power = ofdm.tx_frames(packed, 2, pkg.MODE_EXACT)
    ofdm.replayed_frames(reset=True)
    runs["fast_replay_all"] = (ofdm.awgn_rx_inject_sweep(frames, g, packed, snr, 2, pkg.MODE_FAST, power=power), ofdm.replayed_frames())
    for a, b, c, d, e in zip(runs["fused"][0], runs["replay_all"][0], runs["all_exact"][0], runs["staged_checked"][0], runs["fast_replay_all"][0]):
        assert ints(a) == ints(b) == ints(c) == ints(d) == ints(e)
        assert abs(a.sum_err2 - c.sum_err2) <= 1e-6 * c.sum_err2 and abs(a.sum_evm_lin - c.sum_evm_lin) <= 1e-6 * c.sum_evm_lin
        assert abs(b.sum_err2 - c.sum_err2) <= 1e-7 * c.sum_err2           # the replay is the all-exact kernel's arithmetic (float partial sums grouped differently)
    assert runs["replay_all"][1] == runs["fast_replay_all"][1] == n * len(snr) and runs["all_exact"][1] == 0
    assert 0 < runs["fused"][1] < n * len(snr) // 10                       # speculation must pay


def test_adversarial_frames_through_the_fused_sweep(knobs, pkg, port):
    """frames whose decisions hinge on the reference's rounding, and degenerate draws / frames"""
    ofdm = knobs
    n_frames = 256
    bits, g = bits_and_noise(5, n_frames, 2)
    g[0] = 0.0                                            # no noise at all: sigma N = 0
    g[1, 32:160] = 0.0                                    # clean LTS, noisy data
    g[2] *= np.float32(1e-20)
    g[3] *= np.float32(1e6)
    g[4, 200] = np.float32(3e19)                          # one enormous draw: the window's energy leaves the trusted range
    g[5] = np.float32(1.0)                                # constant draws: all the noise in the DC bin
    g[6, 176:240] = -g[6, 256:320]
    packed = ofdm.to_dev(pkg.pack_bits_host(bits).view(np.int32))
    gd = ofdm.to_dev(g)
    snr = [-10.0, 0.0, 5.0, 20.0, 60.0, 120.0]
    got = ofdm.sweep_inject_dev(packed, gd, n_frames, 2, snr, pkg.MODE_EXACT)
    want = port.chain_sweep(bits, g, 2, snr)
    for s, a, w in zip(snr, got, want):
        assert ints(a) == (w.bit_errors, w.bits, w.frames_in_error, w.rail_errors, w.frames), s


def test_host_route_uses_the_fused_kernel(knobs, pkg, port):
    ofdm = knobs
    n = 70_000                                            # more than one 64 Ki-frame chunk of the host pipeline
    bits, g = bits_and_noise(2, n, 2)
    packed = pkg.pack_bits_host(bits)
    l0 = ofdm.launch_count
    a = ofdm.sweep_inject_host(packed, g, n, 2, SNR21, pkg.MODE_EXACT)
    launches = ofdm.launch_count - l0
    assert launches <= 2 * 3 + 2                          # per chunk: transmitter, power, ONE sweep kernel
    ofdm.set_option("fused_sweep", 0)
    b = ofdm.sweep_inject_host(packed, g, n, 2, SNR21, pkg.MODE_EXACT)
    for x, y in zip(a, b):
        assert ints(x) == ints(y)
    w = port.chain_sweep(bits[:3000], g[:3000], 2, [4.0])[0]
    c = ofdm.sweep_inject_host(packed[:3000], g[:3000], 3000, 2, [4.0], pkg.MODE_EXACT)[0]
    assert ints(c) == (w.bit_errors, w.bits, w.frames_in_error, w.rail_errors, w.frames)
