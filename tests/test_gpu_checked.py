"""OFDM_MODE_EXACT sweeps speculate in fp32, verify every rail decision against a rigorous error bound and replay
doubtful frames in the reference's arithmetic (ofdm_chain.cuh, kArithChecked).  The error counts must be exactly
those of the reference: checked here against the CPU oracle, against the all-exact kernel and against a run in
which every frame is replayed, on ordinary and on adversarial inputs."""
import numpy as np
import pytest

from conftest import bits_and_noise

pytestmark = pytest.mark.gpu


def ints(c):
    return (c.bit_errors, c.bits, c.frames_in_error, c.rail_errors, c.frames)


@pytest.fixture()
def knobs(ofdm):
    """restore the default routing after each test"""
    yield ofdm
    ofdm.set_option("exact_speculation", 1)
    ofdm.set_option("force_replay", 0)
    ofdm.set_option("force_generic_rx", 0)
    ofdm.set_option("stream_layout", 0)
    ofdm.set_option("multipath_path", 0)


# name, arithmetic, exact_speculation, force_replay, force_generic_rx, stream_layout.  The forced replays run every caller of the
# exact replay: one frame per lane group (k_stream_quad), one frame per warp (k_stream_rx2 / k_stream_rxn), and the fp32
# kernels, whose EVM guard replays through the same routine.
VARIANTS = (("checked", "exact", 1, 0, 0, 0), ("all_exact", "exact", 0, 0, 0, 0), ("replay_all", "exact", 1, 1, 0, 0),
            ("replay_all_per_warp", "exact", 1, 1, 0, 1), ("fast_replay_all", "fast", 1, 1, 0, 0),
            ("fast_replay_all_per_warp", "fast", 1, 1, 0, 1), ("generic", "exact", 0, 0, 1, 0))


def run_variants(ofdm, pkg, fn):
    """fn(mode) -> Counters; returns {variant: (Counters, replayed frames)}.  Every forced variant replays every frame and
    gives the all-exact kernel's integer totals."""
    out = {}
    for name, arith, spec, force, generic, layout in VARIANTS:
        ofdm.set_option("exact_speculation", spec)
        ofdm.set_option("force_replay", force)
        ofdm.set_option("force_generic_rx", generic)
        ofdm.set_option("stream_layout", layout)
        ofdm.replayed_frames(reset=True)
        c = fn(pkg.MODE_EXACT if arith == "exact" else pkg.MODE_FAST)
        out[name] = (c, ofdm.replayed_frames())
    ofdm.set_option("stream_layout", 0)
    for name, (c, replayed) in out.items():
        if "replay_all" in name:
            assert ints(c) == ints(out["all_exact"][0]) and replayed == c.frames, name
    return out


@pytest.mark.parametrize("snr", [0.0, 4.0, 9.0, 25.0])
def test_counts_match_oracle_and_all_exact(knobs, pkg, port, snr):
    ofdm = knobs
    n_frames, n_sym = 6000, 2
    bits, g = bits_and_noise(4242 + int(snr), n_frames, n_sym)
    packed = ofdm.to_dev(pkg.pack_bits_host(bits).view(np.int32))
    gd = ofdm.to_dev(g)
    frames, power = ofdm.tx_frames(packed, n_sym, pkg.MODE_EXACT)
    res = run_variants(ofdm, pkg, lambda mode: ofdm.awgn_rx_inject(frames, gd, packed, snr, n_sym, mode, power=power)[0])
    acc = port.chain(bits, g, n_sym, snr)
    want = (acc.bit_errors, acc.bits, acc.frames_in_error, acc.rail_errors, acc.frames)
    for name, (c, _) in res.items():
        assert ints(c) == want, name
        assert abs(c.sum_err2 - acc.sum_err2) <= 1e-5 * acc.sum_err2, name
    assert res["replay_all"][1] == n_frames and res["all_exact"][1] == 0 and res["generic"][1] == 0
    assert res["checked"][1] <= n_frames // 10            # speculation must pay: few replays even at 0 dB
    # the replay runs the all-exact kernel's arithmetic bin by bin: same EVM sums up to the order in which the per-bin
    # float terms of a frame and the per-frame terms of a lane are added up (one frame per lane group vs one per warp)
    a, b = res["replay_all"][0], res["all_exact"][0]
    assert abs(a.sum_err2 - b.sum_err2) <= 1e-6 * b.sum_err2 and abs(a.sum_evm_lin - b.sum_evm_lin) <= 1e-6 * b.sum_evm_lin


def test_large_batch_low_snr(knobs, pkg):
    """300k frames at 0 and 2 dB: thousands of doubtful frames, counts identical to the all-exact kernel"""
    ofdm = knobs
    import torch
    n, n_sym = 300_000, 2
    gen = torch.Generator(device=ofdm.device); gen.manual_seed(99)
    packed = torch.randint(-2**31, 2**31 - 1, (n * 6,), dtype=torch.int32, device=ofdm.device, generator=gen)
    g = torch.randn((n, 320), dtype=torch.float32, device=ofdm.device, generator=gen)
    frames, power = ofdm.tx_frames(packed.view(n, 6), n_sym, pkg.MODE_EXACT)
    for snr in (0.0, 2.0):
        res = run_variants(ofdm, pkg, lambda mode: ofdm.awgn_rx_inject(frames, g, packed, snr, n_sym, mode, power=power)[0])
        want = ints(res["all_exact"][0])
        assert ints(res["checked"][0]) == want and ints(res["replay_all"][0]) == want and ints(res["generic"][0]) == want
        assert 0 < res["checked"][1] < n // 10
        assert abs(res["checked"][0].sum_err2 - res["all_exact"][0].sum_err2) <= 1e-5 * res["all_exact"][0].sum_err2


def rotate_bodies(frames, angle):
    """rotate the data symbols (not the LTS) by `angle`: at 45 degrees every QPSK point lands on a decision boundary"""
    out = frames.copy()
    z = out[:, 160:, 0].astype(np.float32) + 1j * out[:, 160:, 1].astype(np.float32)
    z = (z.astype(np.complex64) * np.complex64(np.exp(1j * angle))).astype(np.complex64)
    out[:, 160:, 0] = z.real; out[:, 160:, 1] = z.imag
    return out


@pytest.mark.parametrize("angle", [np.pi / 4, np.pi / 4 + 3e-7, np.pi / 4 - 2e-5, np.pi / 4 + 1e-3, 3 * np.pi / 4, 0.3])
def test_decisions_on_the_boundary(knobs, pkg, port, angle):
    """noise-free frames whose data bins sit on (or within rounding of) the slicer boundary: the decision is a matter
    of the reference's rounding, bin by bin"""
    ofdm = knobs
    n_frames, n_sym = 400, 2
    bits, _ = bits_and_noise(7, n_frames, n_sym)
    packed = ofdm.to_dev(pkg.pack_bits_host(bits).view(np.int32))
    ota = rotate_bodies(port.tx_frames(bits, n_sym), angle)
    want = port.rx_frames(ota, bits, n_sym)
    od = ofdm.to_dev(ota)
    res = run_variants(ofdm, pkg, lambda mode: ofdm.rx_frames(od, packed, n_sym, mode)[0])
    for name, (c, _) in res.items():
        assert c.bit_errors == int(want["bit_errors"].sum()), name
        assert c.rail_errors == int(want["rail_errors"].sum()), name
        assert c.frames_in_error == int((want["bit_errors"] > 0).sum()), name
    if abs(angle - np.pi / 4) < 1e-6:
        assert res["checked"][1] == n_frames              # nothing on the boundary may be trusted to fp32


def test_degenerate_frames(knobs, pkg, port):
    """zero frames, zero LTS (H = 0 -> the division's recovery branch), denormal-range, huge, NaN and Inf samples"""
    ofdm = knobs
    n_sym = 2
    bits, g = bits_and_noise(21, 64, n_sym)
    tx = port.tx_frames(bits, n_sym)
    rng = np.random.default_rng(5)
    ota = port.awgn_inject(tx, g, 8.0).astype(np.float32)
    ota[0] = 0.0                                          # all-zero capture
    ota[1, :160] = 0.0                                    # no LTS: H = 0 everywhere
    ota[2, 32:96] = -ota[2, 96:160]                       # LTS halves cancel: H = +-0
    ota[3] *= np.float32(1e-30)                           # products underflow
    ota[4] *= np.float32(1e-18)
    ota[5] *= np.float32(1e12)
    ota[6] *= np.float32(3e18)                            # |H|^2 overflows float
    ota[7, 200, 0] = np.nan
    ota[8, 50, 1] = np.inf
    ota[9, 160:] = 0.0                                    # no data
    ota[10] = rng.standard_normal(ota[10].shape).astype(np.float32) * np.float32(1e-22)
    ota[11, 32:160] *= np.float32(1e-6)                   # tiny channel estimate, normal data
    ota[12, 160:] *= np.float32(1e-7)
    finite = [i for i in range(64) if i not in (7, 8)]
    packed = ofdm.to_dev(pkg.pack_bits_host(bits).view(np.int32))
    od = ofdm.to_dev(ota)
    res = run_variants(ofdm, pkg, lambda mode: ofdm.rx_frames(od, packed, n_sym, mode)[0])
    want = ints(res["generic"][0])
    for name, (c, _) in res.items():
        assert ints(c) == want, name
    # against the oracle, frame by frame (the generic kernel's dump path divides exactly)
    w = port.rx_frames(ota, bits, n_sym)
    _, d = ofdm.rx_frames(od, packed, n_sym, pkg.MODE_EXACT, want=("frame_bit_errors",))
    got = d["frame_bit_errors"].cpu().numpy()
    assert np.array_equal(got[finite], w["bit_errors"][finite])
    sel = ofdm.to_dev(ota[finite]); pk = ofdm.to_dev(pkg.pack_bits_host(bits[finite]).view(np.int32))
    ofdm.set_option("exact_speculation", 1); ofdm.set_option("force_replay", 0); ofdm.set_option("force_generic_rx", 0)
    c, _ = ofdm.rx_frames(sel, pk, n_sym, pkg.MODE_EXACT)
    assert c.bit_errors == int(w["bit_errors"][finite].sum()) and c.rail_errors == int(w["rail_errors"][finite].sum())


def test_sweep_entry_points_use_it(knobs, pkg):
    """the sweep entry points give the same totals with and without speculation"""
    ofdm = knobs
    n, n_sym = 50_000, 2
    rng = np.random.default_rng(1)
    bits_h = rng.integers(-2**31, 2**31 - 1, (n, 6), dtype=np.int64).astype(np.int32)
    g_h = rng.standard_normal((n, 320)).astype(np.float32)
    snr = np.arange(0, 21, 4, dtype=np.float32)
    ofdm.replayed_frames(reset=True)
    a = ofdm.sweep_inject_host(bits_h, g_h, n, n_sym, snr, pkg.MODE_EXACT)
    assert ofdm.replayed_frames() > 0
    ofdm.set_option("exact_speculation", 0)
    b = ofdm.sweep_inject_host(bits_h, g_h, n, n_sym, snr, pkg.MODE_EXACT)
    for x, y in zip(a, b):
        assert ints(x) == ints(y)
        assert abs(x.sum_err2 - y.sum_err2) <= 1e-5 * y.sum_err2


def test_error_radius_has_margin(ofdm, pkg, port):
    """The verification trusts |fp32 transform - reference transform| <= 320 u |x|_2 per bin (DESIGN.md section 4).  Measured on
    random, sparse, tonal and wide-dynamic-range inputs the distance stays far inside that radius."""
    rng = np.random.default_rng(77)
    n = 4000
    x = rng.standard_normal((n, 64, 2)).astype(np.float32)
    x[500:1000] *= np.exp(rng.uniform(-20, 20, (500, 1, 1))).astype(np.float32)                     # overall scale
    x[1000:1500] *= np.exp(rng.uniform(-8, 8, (500, 64, 1))).astype(np.float32)                     # per-sample dynamic range
    k = rng.integers(0, 64, 500); t = np.arange(64)
    tone = np.exp(2j * np.pi * k[:, None] * t[None, :] / 64)                                        # single tones: one huge bin
    x[1500:2000, :, 0] = tone.real; x[1500:2000, :, 1] = tone.imag
    x[2000:2500] = 0; x[2000:2500, rng.integers(0, 64, 500), 0] = 1.0                               # impulses
    x[2500:3000, :, 1] = 0                                                                          # real-only
    x[3000:3500] = np.sign(x[3000:3500])                                                            # +-1 patterns
    xd = ofdm.to_dev(x)
    exact = ofdm.fft64(xd, pkg.MODE_EXACT).cpu().numpy().astype(np.float64)
    fast = ofdm.fft64(xd, pkg.MODE_FAST).cpu().numpy().astype(np.float64)
    assert np.array_equal(exact.astype(np.float32), port.fft64(x))                                  # exact = the reference's transform
    err = np.sqrt(((exact - fast) ** 2).sum(axis=2)).max(axis=1)                                    # worst bin per window
    norm = np.sqrt((x.astype(np.float64) ** 2).sum(axis=(1, 2)))
    u = 2.0 ** -24
    assert np.all(err <= 320 * u * norm / 12)                                                       # observed: a few u |x|_2


@pytest.mark.parametrize("snr", [1.0, 7.0])
def test_philox_noise_checked(knobs, pkg, snr):
    """on-chip Philox draws: the replay regenerates the same draws; all routings give the same totals"""
    ofdm = knobs
    import torch
    n, n_sym = 100_000, 2
    gen = torch.Generator(device=ofdm.device); gen.manual_seed(5)
    packed = torch.randint(-2**31, 2**31 - 1, (n * 6,), dtype=torch.int32, device=ofdm.device, generator=gen)
    frames, power = ofdm.tx_frames(packed, n_sym, pkg.MODE_EXACT)
    res = run_variants(ofdm, pkg, lambda mode: ofdm.awgn_rx_philox(frames, packed, snr, 77, 3, 1000, n_sym, mode, power=power)[0])
    want = ints(res["all_exact"][0])
    for name, (c, _) in res.items():
        assert ints(c) == want, name
    assert 0 < res["checked"][1] < n // 10 and res["replay_all"][1] == n


def test_multipath_sweep_checked(knobs, pkg):
    ofdm = knobs
    snr = [2.0, 8.0, 14.0]
    ofdm.set_option("exact_speculation", 1)
    a = ofdm.mc_sweep_multipath(9, 0, 60_000, 2, 6, snr, pkg.MODE_EXACT)
    ofdm.set_option("exact_speculation", 0)
    b = ofdm.mc_sweep_multipath(9, 0, 60_000, 2, 6, snr, pkg.MODE_EXACT)
    # the fused verified kernel (k_mc_philox with taps) with every (frame, point) replayed
    ofdm.set_option("exact_speculation", 1); ofdm.set_option("multipath_path", 2); ofdm.set_option("force_replay", 1)
    ofdm.replayed_frames(reset=True)
    c = ofdm.mc_sweep_multipath(9, 0, 60_000, 2, 6, snr, pkg.MODE_EXACT)
    assert ofdm.replayed_frames() == 60_000 * len(snr)
    for x, y, z in zip(a, b, c):
        assert ints(x) == ints(y) == ints(z)
        assert abs(x.sum_err2 - y.sum_err2) <= 1e-5 * y.sum_err2


def test_monte_carlo_kernel_checked(knobs, pkg):
    """fused on-chip Monte-Carlo in EXACT mode: speculation on / off / forced replay give identical totals"""
    ofdm = knobs
    snr = [float(s) for s in range(-2, 19, 2)]
    n = 150_000
    runs = {}
    # replay_all: k_mc_quad (one frame per lane group); replay_all_per_warp: k_mc_philox
    for name, spec, force, layout in (("checked", 1, 0, 0), ("all_exact", 0, 0, 0), ("replay_all", 1, 1, 0), ("replay_all_per_warp", 1, 1, 1)):
        ofdm.set_option("exact_speculation", spec); ofdm.set_option("force_replay", force); ofdm.set_option("stream_layout", layout)
        ofdm.replayed_frames(reset=True)
        runs[name] = (ofdm.mc_sweep_philox(2024, 5000, n, 2, snr, pkg.MODE_EXACT), ofdm.replayed_frames())
    ofdm.set_option("stream_layout", 0)
    for x, y, z, w in zip(runs["checked"][0], runs["all_exact"][0], runs["replay_all"][0], runs["replay_all_per_warp"][0]):
        assert ints(x) == ints(y) == ints(z) == ints(w)
        assert abs(x.sum_err2 - y.sum_err2) <= 1e-5 * y.sum_err2
        assert abs(z.sum_err2 - y.sum_err2) <= 1e-6 * y.sum_err2          # same per-bin arithmetic, the float terms of a frame added in another order
        assert abs(w.sum_err2 - y.sum_err2) <= 1e-6 * y.sum_err2
    assert runs["replay_all"][1] == runs["replay_all_per_warp"][1] == n * len(snr) and runs["all_exact"][1] == 0
    assert 0 < runs["checked"][1] < n * len(snr) // 10


@pytest.mark.parametrize("n_sym,snr", [(1, 1.0), (3, 5.0), (4, 0.0), (5, 6.0), (6, 2.0), (7, 9.0), (9, 3.0), (23, 4.0)])
def test_other_frame_shapes(knobs, pkg, port, n_sym, snr):
    """frames with n_sym != 2 stream through k_stream_rxn (pass 0 = LTS + two symbols, then four symbols per pass): speculation
    on / off / forced replay, the generic kernel and the oracle agree; fast mode agrees with the generic fast kernel"""
    ofdm = knobs
    n_frames = 1200
    bits, g = bits_and_noise(900 + n_sym, n_frames, n_sym)
    packed = ofdm.to_dev(pkg.pack_bits_host(bits).view(np.int32))
    gd = ofdm.to_dev(g)
    frames, power = ofdm.tx_frames(packed, n_sym, pkg.MODE_EXACT)
    res = run_variants(ofdm, pkg, lambda mode: ofdm.awgn_rx_inject(frames, gd, packed, snr, n_sym, mode, power=power)[0])
    acc = port.chain(bits, g, n_sym, snr)
    want = (acc.bit_errors, acc.bits, acc.frames_in_error, acc.rail_errors, acc.frames)
    for name, (c, _) in res.items():
        assert ints(c) == want, name
        assert abs(c.sum_err2 - acc.sum_err2) <= 1e-5 * acc.sum_err2, name
    assert res["replay_all"][1] == n_frames and res["all_exact"][1] == 0 and res["checked"][1] < n_frames // 2
    for option in (0, 1):
        ofdm.set_option("force_generic_rx", option)
        c = ofdm.awgn_rx_inject(frames, gd, packed, snr, n_sym, pkg.MODE_FAST, power=power)[0]
        if option == 0:
            fast_stream = c
        else:
            assert ints(c) == ints(fast_stream)
    ofdm.set_option("force_generic_rx", 0)
    # noise-free OTA frames and on-chip Philox noise through the same kernel
    ota = ofdm.awgn_inject(frames, gd, snr, n_sym, pkg.MODE_EXACT, power=power)
    a = ofdm.rx_frames(ota, packed, n_sym, pkg.MODE_EXACT)[0]
    assert ints(a) == want
    p1 = ofdm.awgn_rx_philox(frames, packed, snr, 3, 1, 50, n_sym, pkg.MODE_EXACT, power=power)[0]
    ofdm.set_option("force_generic_rx", 1)
    p2 = ofdm.awgn_rx_philox(frames, packed, snr, 3, 1, 50, n_sym, pkg.MODE_EXACT, power=power)[0]
    assert ints(p1) == ints(p2)


def test_general_stream_kernel_on_the_default_shape(knobs, pkg):
    """the multi-pass kernel restricted to pass 0 must reproduce k_stream_rx2 on two-symbol frames"""
    ofdm = knobs
    import torch
    n, n_sym = 200_000, 2
    gen = torch.Generator(device=ofdm.device); gen.manual_seed(12)
    packed = torch.randint(-2**31, 2**31 - 1, (n * 6,), dtype=torch.int32, device=ofdm.device, generator=gen)
    g = torch.randn((n, 320), dtype=torch.float32, device=ofdm.device, generator=gen)
    frames, power = ofdm.tx_frames(packed, n_sym, pkg.MODE_EXACT)
    try:
        for mode in (pkg.MODE_EXACT, pkg.MODE_FAST):
            for snr in (1.0, 9.0):
                ofdm.set_option("general_stream", 0)
                a = ofdm.awgn_rx_inject(frames, g, packed, snr, n_sym, mode, power=power)[0]
                ofdm.set_option("general_stream", 1)
                b = ofdm.awgn_rx_inject(frames, g, packed, snr, n_sym, mode, power=power)[0]
                assert ints(a) == ints(b)
                assert abs(a.sum_err2 - b.sum_err2) <= 1e-6 * b.sum_err2 and abs(a.sum_evm_lin - b.sum_evm_lin) <= 1e-6 * b.sum_evm_lin
    finally:
        ofdm.set_option("general_stream", 0)
