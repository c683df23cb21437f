"""The coded link's CPU oracle (tests/coded_oracle.c, DESIGN.md section 6.2) against independent numpy models written from the
802.11a text: the encoder, the tail, the interleaver, the precoding onto the project's QPSK map, and the Viterbi decoder's
error correction and maximum-likelihood property.  No GPU needed."""
import numpy as np
import pytest

from coded_oracle import CodedOracle, DBPS, correlation, k_info, np_encode, np_viterbi

RATES = ["1/2", "3/4"]


@pytest.fixture(scope="module")
def co():
    return CodedOracle()


def deinterleave_precoded(payload, n_sym):
    """payload bits [n, 96 n_sym] -> the coded bits in transmission order, undoing the precoding and the interleaver"""
    p = payload.reshape(payload.shape[0], n_sym, 48, 2).astype(np.int64)
    c1 = 1 - p[..., 0]
    c0 = p[..., 1] ^ c1
    pos = np.stack([c0, c1], axis=-1).reshape(payload.shape[0], n_sym, 96)
    k = np.arange(96)
    return pos[:, :, 6 * (k % 16) + k // 16].reshape(payload.shape[0], -1)


@pytest.mark.parametrize("rate", RATES)
@pytest.mark.parametrize("n_sym", [1, 2, 5, 512])
def test_encoder_matches_shift_register(co, rate, n_sym):
    rng = np.random.default_rng(n_sym)
    n = 2 if n_sym == 512 else 16
    info = rng.integers(0, 2, (n, 96 * n_sym), dtype=np.uint8)
    payload = co.conv_encode(info, n_sym, rate)
    assert np.array_equal(deinterleave_precoded(payload, n_sym), np_encode(info, rate, n_sym))
    # bits beyond K_info (the tail's slot and the unused rest of the words) do not matter
    info2 = info.copy()
    info2[:, k_info(rate, n_sym):] ^= 1
    assert np.array_equal(co.conv_encode(info2, n_sym, rate), payload)


def test_impulse_response_and_tail(co):
    n_sym = 2
    info = np.zeros((1, 192), np.uint8)
    info[0, 0] = 1
    coded = np_encode(info, "1/2", n_sym)[0]
    assert coded.sum() == 10                                    # free distance of the K = 7 code: the impulse response's weight
    assert np.array_equal(deinterleave_precoded(co.conv_encode(info, n_sym, "1/2"), n_sym)[0], coded)
    # the tail returns the encoder to state 0: the last 6 steps of any frame see zero inputs, so the coded stream of the
    # frame's last information bits is that of a frame that ends right after them
    rng = np.random.default_rng(3)
    info = rng.integers(0, 2, (8, 192), dtype=np.uint8)
    K = k_info("1/2", n_sym)
    T = n_sym * 48
    x = np.zeros((8, T + 6), np.int64)
    x[:, 6:6 + K] = info[:, :K]
    assert not x[:, T:].any()                                    # the last window (x[T-1] .. x[T-6]) is all zero: state 0


def test_interleaver_formula(co):
    pos = [co.interleave(k) for k in range(96)]
    assert sorted(pos) == list(range(96))                      # a permutation
    # 802.11a 17.3.5.6: i = (N_CBPS / 16)(k mod 16) + floor(k / 16); j = s floor(i / s) + (i + N_CBPS - floor(16 i / N_CBPS)) mod s
    # with s = max(N_BPSC / 2, 1) = 1 for QPSK: j = i
    for k in range(96):
        i = (96 // 16) * (k % 16) + k // 16
        assert pos[k] == i and 1 * (i // 1) + (i + 96 - (16 * i) // 96) % 1 == i


def test_precoding_gives_the_80211a_constellation(co):
    q = np.float32(1.0 / np.sqrt(2.0))
    for c0 in (0, 1):
        for c1 in (0, 1):
            bits = np.zeros(96, np.uint8)
            bits[0], bits[1] = 1 - c1, c0 ^ c1                   # (a, b) = (!c1, c0 ^ c1)
            p = co.qpsk_mod(bits, 1)[0]
            assert p[0] == (2 * c0 - 1) * q and p[1] == (2 * c1 - 1) * q, (c0, c1, p)


def clean_inputs(payload, n_sym):
    """H = 1 on every bin and eq = the noise-free constellation of the payload bits"""
    n = payload.shape[0]
    H = np.zeros((n, 64, 2), np.float32)
    H[..., 0] = 1.0
    p = payload.reshape(n, n_sym * 48, 2).astype(np.int64)
    c1 = 1 - p[..., 0]
    c0 = p[..., 1] ^ c1
    eq = np.stack([2 * c0 - 1, 2 * c1 - 1], axis=-1).astype(np.float32) / np.float32(np.sqrt(2.0))
    return H, eq


@pytest.mark.parametrize("rate", RATES)
@pytest.mark.parametrize("decision", ["soft", "hard"])
def test_viterbi_noise_free(co, rate, decision):
    rng = np.random.default_rng(11)
    for n_sym in (1, 2, 7):
        info = rng.integers(0, 2, (12, 96 * n_sym), dtype=np.uint8)
        H, eq = clean_inputs(co.conv_encode(info, n_sym, rate), n_sym)
        assert np.array_equal(co.viterbi(H, eq, n_sym, rate, decision), info[:, :k_info(rate, n_sym)])


@pytest.mark.parametrize("rate,max_flips", [("1/2", 4), ("3/4", 2)])
def test_viterbi_corrects_up_to_half_the_free_distance(co, rate, max_flips):
    rng = np.random.default_rng(5)
    n_sym = 3
    for trial in range(60):
        info = rng.integers(0, 2, (1, 96 * n_sym), dtype=np.uint8)
        H, eq = clean_inputs(co.conv_encode(info, n_sym, rate), n_sym)
        flips = rng.choice(n_sym * 96, size=int(rng.integers(1, max_flips + 1)), replace=False)
        eq.reshape(-1)[flips] *= -1                               # hard errors on single rails (coded bits)
        for decision in ("soft", "hard"):
            assert np.array_equal(co.viterbi(H, eq, n_sym, rate, decision), info[:, :k_info(rate, n_sym)]), (rate, trial, flips)


@pytest.mark.parametrize("rate", RATES)
def test_viterbi_is_maximum_likelihood(co, rate):
    """on random soft inputs the oracle's path has the float64 correlation of the numpy model's best path (fp32 metrics)"""
    rng = np.random.default_rng(17)
    n_sym, n = 2, 40
    H = np.zeros((n, 64, 2), np.float32)
    H[..., 0] = 1.0
    eq = rng.standard_normal((n, n_sym * 48, 2)).astype(np.float32)
    dec = co.viterbi(H, eq, n_sym, rate, "soft")
    from coded_oracle import np_inputs
    La, Lb = np_inputs(H, eq, n_sym, rate, "soft")
    _, best = np_viterbi(La, Lb)
    info = np.zeros((n, 96 * n_sym), np.uint8)
    info[:, :dec.shape[1]] = dec
    # re-encode the oracle's decision (tail included) and correlate in float64
    ab = np_encode(info, rate, n_sym)
    for f in range(n):
        got = correlation(ab[f], La[f], Lb[f], rate)
        assert abs(got - best[f]) <= 1e-6 * abs(best[f]), (f, got, best[f])
    assert DBPS[rate] * n_sym - 6 == dec.shape[1]
