"""CPU checks of the channel definitions (ofdm_channel, DESIGN.md "Channels"): the draws, the channel oracle against the pinned
oracle, the oracle's whole chain against an independent float64 model, and the textbook curve sweep.qpsk_ber_awgn."""
import numpy as np
import pytest

from channel_oracle import DOMAIN_NOISE, DOMAIN_NOISE_Q, ChannelOracle, model_complex_esn0


@pytest.fixture(scope="module")
def co():
    return ChannelOracle()


def test_domain4_draws_and_i_rail_identity(co, port):
    L = co.frame_len(2)
    g0 = co.philox_normals(11, 3, 1000, 64, L, DOMAIN_NOISE)
    g1 = co.philox_normals(11, 3, 1000, 64, L, DOMAIN_NOISE_Q)
    assert np.array_equal(g0, port.philox_normals(11, 3, 1000, 64, L))       # domain 0 = the pinned oracle's noise draws
    assert not np.any(g0 == g1)
    assert abs(np.corrcoef(g0.ravel(), g1.ravel())[0, 1]) < 0.02
    # the complex channel's I rail carries exactly the domain-0 draws, the Q rail the domain-4 ones
    tx = co.tx_frames(co.philox_bits(11, 1000, 64, 2), 2)
    out = co.awgn_channel(tx, g0, g1, 3.0, "complex", "esn0")
    np_ = np.float32(1.0 / (64.0 * 10.0 ** 0.3))
    sigma = np.sqrt(0.5 * np.float64(np_))
    assert np.array_equal(out[..., 0], (tx[..., 0] + (sigma * g0.astype(np.float64)).astype(np.float32)).astype(np.float32))
    assert np.array_equal(out[..., 1], (tx[..., 1] + (sigma * g1.astype(np.float64)).astype(np.float32)).astype(np.float32))


def test_reference_channel_and_rail_variances(co, port):
    rng = np.random.default_rng(5)
    n_sym = 3
    bits = rng.integers(0, 2, (40, 96 * n_sym), dtype=np.uint8)
    tx = co.tx_frames(bits, n_sym)
    g0 = rng.standard_normal((40, co.frame_len(n_sym))).astype(np.float32)
    g1 = rng.standard_normal((40, co.frame_len(n_sym))).astype(np.float32)
    for snr in (-3.0, 6.0, 21.5):
        assert np.array_equal(co.awgn_channel(tx, g0, None, snr, "real", "frame_power"), port.awgn_inject(tx, g0, snr))
    # complex noise: total variance np, half per rail, for every SNR definition
    g0 = co.philox_normals(2, 0, 0, 4000, co.frame_len(n_sym), DOMAIN_NOISE)
    g1 = co.philox_normals(2, 0, 0, 4000, co.frame_len(n_sym), DOMAIN_NOISE_Q)
    tx = np.zeros((4000, co.frame_len(n_sym), 2), np.float32)
    for snr_def, per_point in (("esn0", 64.0), ("ebn0", 128.0)):
        np_ = 1.0 / (per_point * 10.0 ** 0.5)
        d = co.awgn_channel(tx, g0, g1, 5.0, "complex", snr_def).astype(np.float64)
        for rail in (0, 1):
            assert abs(d[..., rail].var() / (np_ / 2) - 1.0) < 0.01, (snr_def, rail)
        r = co.awgn_channel(tx, g0, None, 5.0, "real", snr_def).astype(np.float64)
        assert abs(r[..., 0].var() / np_ - 1.0) < 0.01 and not r[..., 1].any()


def _mean_and_var(per_frame):
    x = np.asarray(per_frame, dtype=np.float64)
    return x.mean(), x.var(ddof=1) / len(x)


def test_oracle_chain_matches_independent_model(co):
    """orc_chain_channel (complex / Es/N0, on the Philox draws) against the float64 model: BER and frame error rate agree within
    4 combined standard errors; the variances come from per-frame counts (a frame's errors share its channel estimate)."""
    n_frames, n_sym = 20000, 2
    rng = np.random.default_rng(123)
    for i, snr in enumerate((0.0, 2.0, 4.0, 6.0)):
        acc, fe, _ = co.mc_sweep(9, 0, n_frames, n_sym, [snr], "complex", "esn0", streams=[i], per_frame=True)[0]
        assert int(acc.bit_errors) == int(fe.sum()) and acc.frames == n_frames
        model = model_complex_esn0(snr, n_frames, n_sym, rng)
        for stat in (lambda e: e / (96.0 * n_sym), lambda e: (e > 0).astype(np.float64)):
            ma, va = _mean_and_var(stat(fe.astype(np.float64)))
            mb, vb = _mean_and_var(stat(model.astype(np.float64)))
            assert abs(ma - mb) <= 4.0 * np.sqrt(va + vb), (snr, ma, mb, np.sqrt(va + vb))


def test_qpsk_ber_awgn_against_simulation(pkg):
    rng = np.random.default_rng(77)
    n = 2_000_000
    for snr in (0.0, 3.0, 6.0):
        for snr_def in ("esn0", "ebn0"):
            esn0 = 10.0 ** (snr / 10.0) * (2.0 if snr_def == "ebn0" else 1.0)
            sigma = np.sqrt(1.0 / (2.0 * esn0))             # per rail, |X| = 1
            ei = rng.standard_normal(n) * sigma < -1.0 / np.sqrt(2.0)
            eq = rng.standard_normal(n) * sigma < -1.0 / np.sqrt(2.0)
            per_sym = np.where(ei & eq, 1, ei * 1 + eq * 2)
            m, v = _mean_and_var(per_sym / 2.0)
            want = float(pkg.sweep.qpsk_ber_awgn(snr, snr_def))
            assert abs(m - want) <= 4.0 * np.sqrt(v), (snr, snr_def, m, want)
    assert pkg.sweep.qpsk_ber_awgn([0.0, 10.0], "esn0")[1] < pkg.sweep.qpsk_ber_awgn([0.0, 10.0], "esn0")[0]
    with pytest.raises(ValueError):
        pkg.sweep.qpsk_ber_awgn(3.0, "frame_power")


def test_channel_names(pkg):
    ch = pkg.channel("complex", "ebn0", 4)
    assert (ch.noise, ch.snr_def, ch.n_taps) == (1, 2, 4)
    assert (pkg.channel().noise, pkg.channel().snr_def, pkg.channel().n_taps) == (0, 0, 0)
    for bad in (dict(noise="imag"), dict(snr_def="snr")):
        with pytest.raises(ValueError):
            pkg.channel(**bad)
